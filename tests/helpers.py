"""Shared helpers for the parity tests (test infrastructure)."""
from __future__ import annotations

import numpy as np
import torch

from oracle import OracleAgent, OracleHps
from tests.golden.cases import case_inputs


def rel_dev(a, b, scale=None) -> float:
    """max|a-b| / max|b| — the per-tensor tolerance definition of BASELINE.md §4.6.
    ``scale`` replaces the denominator for scalars that are a difference of large terms."""
    a = torch.as_tensor(a).detach().to("cpu", torch.float64)
    b = torch.as_tensor(b).detach().to("cpu", torch.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    denom = float(scale) if scale is not None else max(float(b.abs().max()), 1e-30)
    return float((a - b).abs().max()) / denom


def oracle_hps(h: dict, capturable: bool = False) -> OracleHps:
    f = OracleHps.__dataclass_fields__
    return OracleHps(**{k: v for k, v in h.items() if k in f}, adam_capturable=capturable)


def make_oracle(inp, dtype=torch.float32, capturable=True) -> OracleAgent:
    cast = lambda d: {k: v.to(dtype) for k, v in d.items()}
    return OracleAgent(inp["ob"], inp["ac"], inp["min_ac"], inp["max_ac"], oracle_hps(inp["hps"], capturable),
                       dtype=dtype, actor_init=cast(inp["actor"]), qnet_init=[cast(inp["q1"]), cast(inp["q2"])])


def oracle_cuda(inp, dtype) -> OracleAgent:
    """The reference learner on the GPU (float32 or float64) with the case's parameters. Its fp32 products must be
    true fp32: on TF32 the fp32 oracle would be a worse yardstick than the CUDA path it judges."""
    assert not torch.backends.cuda.matmul.allow_tf32 and torch.get_float32_matmul_precision() == "highest", \
        "the fp32 oracle must not run its products on TF32"
    cast = lambda d: {k: v.to(dtype) for k, v in d.items()}
    return OracleAgent(inp["ob"], inp["ac"], inp["min_ac"], inp["max_ac"], oracle_hps(inp["hps"], True), device="cuda", dtype=dtype,
                       actor_init=cast(inp["actor"]), qnet_init=[cast(inp["q1"]), cast(inp["q2"])])


def make_agent(inp, device="cuda", seed=0):
    from sac_td3_cudagraphs_pytorch_b200 import Hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    ag = Agent({"ob_shape": (inp["ob"],), "ac_shape": (inp["ac"],)}, inp["min_ac"], inp["max_ac"],
               torch.device(device), Hps(inp["hps"]), rb=None, seed=seed)
    ag.load_params(inp["actor"], inp["q1"], inp["q2"])
    return ag


def batch_of(inp, i, dtype=torch.float32, device="cpu"):
    idx = inp["idx"][i]
    return {k: (v[idx].to(dtype) if v.is_floating_point() else v[idx]).to(device) for k, v in inp["storage"].items()}


def alpha_loss_scale(alpha, ac_dim) -> float:
    """alpha_loss = alpha * (mean(-logpi) - targ_ent) with targ_ent = -A is a difference of two O(A)
    terms (it crosses zero as the entropy reaches its target), so its error is judged against
    alpha * A, the size of the terms, not against the cancelled result."""
    return float(alpha) * float(ac_dim)


def check_close(name, got, ref32, ref64, floor=1e-5, factor=4.0, scale=None):
    """CUDA result vs the fp32 oracle, with the fp32 oracle's own distance to float64 as yardstick:
    dev(cuda, fp32) <= max(floor, factor * dev(fp32, fp64)). Returns the three numbers for reporting."""
    d_cuda = rel_dev(got, ref32, scale)
    d_ref = rel_dev(ref32, ref64, scale)
    d_true = rel_dev(got, ref64, scale)
    tol = max(floor, factor * d_ref)
    assert d_cuda <= tol or d_true <= tol, (
        f"{name}: cuda-vs-oracle32 {d_cuda:.3e}, cuda-vs-oracle64 {d_true:.3e}, "
        f"oracle32-vs-oracle64 {d_ref:.3e}, tol {tol:.3e}")
    return d_cuda, d_true, d_ref


def check_param_after_first_adam(name, got, ref32, ref64, g_got, g_ref32, lr, floor=1e-5, factor=4.0, adam_eps=1e-8):
    """Parameter check after the FIRST Adam step (zero moments), element-wise.

    The first Adam step is p -= lr * g / (|g| + eps): for an element whose gradient is ~1e-7 the update is
    a steep function of g, so two correct fp32 gradients that differ by 2e-9 (3e-8 of max|g|, far inside the
    gradient tolerance) move the parameter differently by ~1e-6 — measured on sac_humanoid fc_block_2.fc.weight
    [5797]: g = -7.25e-8 (CUDA) vs -7.48e-8 (torch fp32) vs -7.49e-8 (float64). The allowance is therefore
    the usual relative bound on the tensor PLUS, per element, the exact difference of the Adam update ratios
    of the two gradients (which the gradient check has already bounded); nothing else is forgiven."""
    got = torch.as_tensor(got).detach().to("cpu", torch.float64)
    r32 = torch.as_tensor(ref32).detach().to("cpu", torch.float64)
    r64 = torch.as_tensor(ref64).detach().to("cpu", torch.float64)
    g1 = torch.as_tensor(g_got).detach().to("cpu", torch.float64)
    g2 = torch.as_tensor(g_ref32).detach().to("cpu", torch.float64)
    ratio = lambda g: g / (g.abs() + adam_eps)
    tol = max(floor, factor * rel_dev(r32, r64))
    allowed = tol * float(r32.abs().max()) + 1.01 * lr * (ratio(g1) - ratio(g2)).abs()
    excess = ((got - r32).abs() - allowed).max()
    assert float(excess) <= 0.0, (
        f"{name}: |cuda - oracle32| exceeds tol*max|p| + lr*|adam_ratio(g_cuda) - adam_ratio(g_oracle32)| by "
        f"{float(excess):.3e} (plain rel dev {rel_dev(got, r32):.3e}, tol {tol:.3e})")


def kink_safe(inp, batch, margin=2e-5):
    """Rows of the batch whose online-critic pre-activations all stay `margin` away from the ReLU kink.
    The update is discontinuous there: a pre-activation of 1.3e-6 (fp32 path, oracle) against <= 0 (3xTF32 path,
    1e-6 away) flips one unit of one row and moves the batch gradient by 1e-2 of its max (measured on td3_hopper,
    critic 1, row 90) — both evaluations are correct to fp32 rounding. Parity is therefore asserted on the rows
    where the comparison is well-posed (a ragged batch, which the wide path takes as it comes)."""
    x = torch.cat([batch["observations"], batch["actions"]], 1).double()
    ok = torch.ones(x.shape[0], dtype=torch.bool, device=x.device)
    ln = bool(inp["hps"]["layer_norm"])
    for q in (inp["q1"], inp["q2"]):
        h = x
        for blk in ("fc_block_1", "fc_block_2"):
            w = lambda k: q[f"fc_stack.{blk}.{k}"].to(x.device, torch.float64)
            z = h @ w("fc.weight").T + w("fc.bias")
            if ln:
                z = (z - z.mean(1, keepdim=True)) / torch.sqrt(z.var(1, unbiased=False, keepdim=True) + 1e-5)
                z = z * w("ln.weight") + w("ln.bias")
            ok &= z.abs().min(1).values > margin
            h = torch.relu(z)
    return ok


def kink_safe_actor(inp, batch, eps, margin=2e-5):
    """As kink_safe, for the actor step: the actor's own layers on obs and the critics' layers on (obs, a_pi)."""
    ob = batch["observations"].double()
    dev = ob.device
    ok = torch.ones(ob.shape[0], dtype=torch.bool, device=dev)
    ln = bool(inp["hps"]["layer_norm"])

    def trunk(x, q):
        nonlocal ok
        h = x
        for blk in ("fc_block_1", "fc_block_2"):
            w = lambda k: q[f"fc_stack.{blk}.{k}"].to(dev, torch.float64)
            z = h @ w("fc.weight").T + w("fc.bias")
            if ln:
                z = (z - z.mean(1, keepdim=True)) / torch.sqrt(z.var(1, unbiased=False, keepdim=True) + 1e-5)
                z = z * w("ln.weight") + w("ln.bias")
            ok &= z.abs().min(1).values > margin
            h = torch.relu(z)
        return h

    a = inp["actor"]
    u = trunk(ob, a) @ a["head.weight"].to(dev, torch.float64).T + a["head.bias"].to(dev, torch.float64)
    lo, hi = torch.as_tensor(inp["min_ac"]).to(dev, torch.float64), torch.as_tensor(inp["max_ac"]).to(dev, torch.float64)
    scale, bias = (hi - lo) / 2, (hi + lo) / 2
    A = inp["ac"]
    if inp["hps"]["prefer_td3_over_sac"]:
        act = torch.tanh(u) * scale + bias
    else:
        ls = -5.0 + 3.5 * (torch.tanh(u[:, A:]) + 1.0)
        act = torch.tanh(u[:, :A] + eps.to(dev, torch.float64) * torch.exp(ls)) * scale + bias
    x = torch.cat([ob, act], 1)
    trunk(x, inp["q1"])
    trunk(x, inp["q2"])
    return ok
