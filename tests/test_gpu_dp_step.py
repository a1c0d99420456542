"""DataParallelLearner's environment-facing step (step_async / wait / wait_actions) and the behaviour policy on the tensor
cores (wide.WidePredictor, b2rl_wide_actor_predict).

Bounds of the wide policy against a float64 forward pass (tests/test_gpu_noise.py policy_ref / check_policy: |got - want|
<= atol + rtol (|want| + |d action / d z * z|)):
  - 3xTF32 rtol = atol = 1e-5, fp32 level: the row kernel's own rtol (its atol is 2e-6). Measured on a B200, the wide
    policy's worst |da| grows with the first layer's fan-in: 2e-6 (mode 0) and 5e-6 (SAC sample, which carries the
    log-std's error times 3.5 through the squash) with 11 inputs; 7e-6 and 1.1e-5 with Humanoid's 376.
  - TF32 rtol = atol = 1e-2: two TF32 products of ~1e-3 each, through LayerNorm and the head."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions
from tests.test_gpu_noise import check_policy, policy_ref

REPO = Path(__file__).resolve().parent.parent
M64 = 2 ** 64 - 1
WIDE_TOL = {"3xtf32": (1e-5, 1e-5), "tf32": (1e-2, 1e-2)}  # (rtol, atol)


def _agent(kind, ob, A, seed=7, agent_id=0, lo=None, hi=None, **over):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    torch.manual_seed(0)
    hps = (sac_hps if kind == "sac" else td3_hps)(**over)
    lo = np.full(A, -1.0, np.float32) if lo is None else np.asarray(lo, np.float32)
    hi = np.full(A, 1.0, np.float32) if hi is None else np.asarray(hi, np.float32)
    return Agent({"ob_shape": (ob,), "ac_shape": (A,)}, lo, hi, torch.device("cuda"), hps, rb=None, seed=seed, agent_id=agent_id)


def _row_predict(ag, obs, mode, eps_out=None):
    """b2rl_actor_predict with the in-graph key (draw = UINT64_MAX: counters[CTR_Q] | 2^31); eps_out records its noise."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    a = L.UpdateArgs()
    a.hp, a.fmt, a.actor = ag._hyper, ag.fmt, ag.layout.actor.c_struct()
    a.arena, a.region_stride, a.agent_base = ag.arena.flat.data_ptr(), ag.layout.region, ag.agent_id
    a.min_ac, a.max_ac, a.counters = ag.min_ac.data_ptr(), ag.max_ac.data_ptr(), ag.counters.data_ptr()
    a.eps_out = L.ptr(eps_out)
    act = torch.empty(obs.shape[0], ag.ac_dim, device="cuda")
    std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
    L.check(ag._lib.b2rl_actor_predict(C.byref(a), obs.data_ptr(), obs.shape[0], mode, std, C.c_uint64(M64), act.data_ptr(),
                                       torch.cuda.current_stream().cuda_stream), "actor_predict")
    return act


def _actor_params(ag):
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    return {k: v.detach().clone() for k, v in ag.arena.named(ag.layout.actor, L.REGION_P).items()}


def test_wide_predict_struct_matches_the_c_compiler():
    """The ctypes mirror of b2rl_wide_predict_t has the C compiler's size and field offsets (no GPU)."""
    import tempfile
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    fields = [f for f, _ in L.WidePredict._fields_]
    src = '#include <stdio.h>\n#include <stddef.h>\n#include "b2rl.h"\nint main(){printf("%zu", sizeof(b2rl_wide_predict_t));' + \
        "".join(f'printf(" %zu", offsetof(b2rl_wide_predict_t, {f}));' for f in fields) + "return 0;}"
    with tempfile.TemporaryDirectory() as d:
        c = Path(d) / "s.c"
        c.write_text(src)
        subprocess.check_call(["gcc", "-I", str(REPO / "include"), str(c), "-o", str(Path(d) / "s")])
        out = [int(x) for x in subprocess.check_output([str(Path(d) / "s")]).split()]
    assert out == [C.sizeof(L.WidePredict)] + [getattr(L.WidePredict, f).offset for f in fields]


# ------------------------------------------------------------------------------------------------ 1. the wide policy
@pytest.mark.gpu
@pytest.mark.parametrize("ob,A", [(11, 3), (17, 6), (376, 17)])
@pytest.mark.parametrize("kind", ["sac", "td3"])
def test_wide_policy_noise_equals_row_predict(kind, ob, A):
    """b2rl_wide_actor_predict after tc_first / tc_linear on n in {1, 4, 130, 4096} rows: its recorded noise is bitwise
    b2rl_actor_predict's in-graph draw; modes 0 and 1 are within the stated bound of a float64 forward pass on the same
    (perturbed) parameters, in 3xTF32 and TF32."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.wide import WidePredictor
    gen = torch.Generator().manual_seed(ob * 100 + A)
    lo, hi = -0.5 - torch.rand(A, generator=gen), 0.2 + 1.5 * torch.rand(A, generator=gen)
    ag = _agent(kind, ob, A, seed=0xC0FFEE123, agent_id=5, lo=lo.numpy(), hi=hi.numpy())
    actor = _actor_params(ag)
    for k, v in actor.items():  # non-trivial biases and LayerNorm affine parameters (the init has zeros / ones)
        if k.endswith("bias"):
            v += 0.1 * torch.randn(v.shape, generator=gen).cuda()
        elif ".ln.weight" in k:
            v += 0.2 * torch.randn(v.shape, generator=gen).cuda()
    with torch.no_grad():
        for k, v in ag.arena.named(ag.layout.actor, L.REGION_P).items():
            v.copy_(actor[k])
    ag.arena.sync_shadows()
    ag.refresh_lo()
    ag.counters[L.CTR_Q] = (1 << 32) * 3 + 41
    std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
    lo_d, hi_d = ag.min_ac.double(), ag.max_ac.double()
    obs_all = torch.randn(4096, ob, generator=gen).cuda()
    ln = bool(ag.hps.layer_norm)
    want0, _ = policy_ref(actor, obs_all, A, ag.td3, ln, lo_d, hi_d, std)
    for prec in ("3xtf32", "tf32"):
        rtol, atol = WIDE_TOL[prec]
        for n in (1, 4, 130, 4096):
            obs = obs_all[:n].contiguous()
            tag = f"{kind} ob={ob} A={A} {prec} n={n}"
            z_row, z_wide = torch.full((n, A), float("nan"), device="cuda"), torch.full((n, A), float("nan"), device="cuda")
            a_row = _row_predict(ag, obs, 1, eps_out=z_row)
            pol = WidePredictor(ag, n, prec)
            a0, a1 = torch.empty(n, A, device="cuda"), torch.empty(n, A, device="cuda")
            pol.enqueue(obs.data_ptr(), False, a0.data_ptr())
            pol.enqueue(obs.data_ptr(), True, a1.data_ptr(), eps_out=z_wide)
            torch.cuda.synchronize()
            assert torch.isfinite(z_row).all() and torch.equal(z_row, z_wide), f"{tag}: noise differs from the row kernel's"
            check_policy(f"wide {tag} mode 0", a0, want0[:n], rtol=rtol, atol=atol)
            want1, dadz = policy_ref(actor, obs, A, ag.td3, ln, lo_d, hi_d, std, z_wide.double())
            check_policy(f"wide {tag} mode 1", a1, want1, dadz, z_wide.double(), rtol=rtol, atol=atol)
            check_policy(f"row {tag} mode 1", a_row, want1, dadz, z_row.double())  # (the row kernel's own bound)


# ------------------------------------------------------------------------------------------------ 2-4. the step
def _learner(kind, wide, policy=None, B=512, cap=3000, fill=2000, graphs=None, agent_id=0, comm=None):
    from sac_td3_cudagraphs_pytorch_b200.dp import DataParallelLearner
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    ag = _agent(kind, 11, 3, agent_id=agent_id, batch_size=B)
    rb = ReplayBuffer(cap, "cuda", seed=9, agent_id=agent_id)
    td = make_synthetic_transitions(fill, 11, 3, [-1.0] * 3, [1.0] * 3, seed=40 + agent_id)
    rb.extend({k: v.cuda() for k, v in td.items()})
    return DataParallelLearner(ag, rb, B, comm, wide=wide, graphs=graphs, policy=policy)


def _inputs(t, n_new, n_obs, fmt, salt=0):
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    rows = torch.zeros(0, fmt.row_stride)
    if n_new:
        rows = pack_rows(make_synthetic_transitions(n_new, 11, 3, [-1.0] * 3, [1.0] * 3, seed=1000 + 17 * t + salt), fmt)
    obs = torch.randn(n_obs, 11, generator=torch.Generator().manual_seed(2000 + t + salt))
    return rows, obs


def _state(dp):
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ag, rb = dp.agent, dp.rb
    return {"arena PTMV": ag.arena.flat[:, L.REGION_P:L.REGION_V + 1].clone(), "counters Q PI ALPHA SAMPLE": ag.counters[:4].clone(),
            "alpha_state": ag._alpha_state[[0, 2, 3]].clone(), "replay": rb.storage.clone(),
            "cursor / size": (rb._cursor, rb._size), "updates": (ag.qnet_updates_so_far, ag.actor_updates_so_far)}


def _assert_same(a, b, what):
    for k in a:
        same = torch.equal(a[k], b[k]) if isinstance(a[k], torch.Tensor) else a[k] == b[k]
        assert same, f"{what}: {k} differs"


CASES = [("sac", None, "row"), ("td3", None, "row"), ("sac", "3xtf32", "row"), ("td3", "3xtf32", "row"),
         ("sac", "3xtf32", "wide"), ("td3", "3xtf32", "wide")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,wide,policy", CASES)
def test_dp_step_equals_eager_extend_predict_iteration(kind, wide, policy):
    """W = 1: step(i, n_new, n_obs, explore) for 3 x (delay + 1) steps against the eager sequence on a clone — row
    b2rl_actor_predict (draw = UINT64_MAX) with the parameters before the step, rb.extend, iteration(i) without graphs:
    arena regions P T M V, counters, alpha state, replay storage / cursor / size and every log block bitwise equal; the
    row policy's actions bitwise, the wide policy's within WIDE_TOL of float64 on the same parameters and noise."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    dp, ref = _learner(kind, wide, policy), _learner(kind, wide, "row", graphs=False)
    assert dp.graphs and not ref.graphs and dp.policy == policy
    ag, T = dp.agent, 3 * (int(dp.agent.hps.actor_update_delay) + 1)
    rtol, atol = WIDE_TOL["3xtf32"]
    std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
    for t in range(T):
        n_new, n_obs, explore = (64, 200, t % 3 != 1) if t != 4 else (0, 0, True)
        rows, obs = _inputs(t, n_new, n_obs, ag.fmt)
        if n_new:
            dp.host_rows(n_new).copy_(rows)
        if n_obs:
            dp.host_obs(n_obs).copy_(obs)
        logs = dp.step(t, n_new, n_obs, explore).clone()
        acts = torch.from_numpy(dp.wait_actions().copy()) if n_obs else None
        # the eager sequence
        if n_obs:
            params = _actor_params(ref.agent)
            z = torch.zeros(n_obs, 3, device="cuda")
            want = _row_predict(ref.agent, obs.cuda(), int(explore), eps_out=z).cpu()
        if n_new:
            ref.rb.extend_rows(rows.cuda())
        ref.iteration(t)
        torch.cuda.synchronize()
        assert torch.equal(logs, ref.agent.out.cpu()), f"step {t}: log block"
        if n_obs and policy == "row":
            assert torch.equal(acts, want), f"step {t}: actions"
        elif n_obs:
            lo_d, hi_d = ag.min_ac.double(), ag.max_ac.double()
            zd = z.double() if explore else None
            w64, dadz = policy_ref(params, obs.cuda(), 3, ag.td3, bool(ag.hps.layer_norm), lo_d, hi_d, std, zd)
            check_policy(f"step {t} wide actions", acts, w64, dadz, zd, rtol=rtol, atol=atol)
    _assert_same(_state(dp), _state(ref), f"{kind} wide={wide} policy={policy}")
    assert ag.counters[L.CTR_CURSOR] == dp.rb._cursor and ag.counters[L.CTR_SIZE] == dp.rb._size
    dp.iteration(T)  # a later iteration() uploads no stale fill count over the one the steps advanced
    ref.iteration(T)
    torch.cuda.synchronize()
    _assert_same(_state(dp), _state(ref), "iteration after the steps")


@pytest.mark.gpu
@pytest.mark.parametrize("kind,wide,policy", [("sac", "3xtf32", "wide"), ("td3", None, "row")])
def test_pipelined_dp_steps_equal_synchronous_steps(kind, wide, policy):
    """Two steps in flight (inputs of step t + 1 staged while step t runs, after waiting for step t - 1) give bitwise the
    results of step() each time: state, every log block, every action. A third step_async waits for the oldest."""
    a, b = _learner(kind, wide, policy), _learner(kind, wide, policy)
    logs_a, logs_b, acts_a, acts_b = [], [], [], []
    for t in range(8):
        rows, obs = _inputs(t, 32, 256, a.agent.fmt)
        a.host_rows(32).copy_(rows)
        a.host_obs(256).copy_(obs)
        logs_a.append(a.step(t, 32, 256).clone())
        acts_a.append(a.wait_actions().copy())
    prev = None
    for t in range(8):
        rows, obs = _inputs(t, 32, 256, b.agent.fmt)
        b.host_rows(32).copy_(rows)
        b.host_obs(256).copy_(obs)
        tk = b.step_async(t, 32, 256)
        acts_b.append(b.wait_actions().copy())
        if prev is not None:
            logs_b.append(b.wait(prev).clone())
        prev = tk
    logs_b.append(b.wait(prev).clone())
    torch.cuda.synchronize()
    _assert_same(_state(a), _state(b), "pipelined vs synchronous")
    assert all(torch.equal(x, y) for x, y in zip(logs_a, logs_b)) and len(logs_b) == 8
    assert all(np.array_equal(x, y) for x, y in zip(acts_a, acts_b))
    t1, t2 = b.step_async(8), b.step_async(9)
    assert b._stage.waited < t1
    b.step_async(10)
    assert b._stage.waited == t1  # (the third waited for the oldest: its staging slot is about to be reused)
    b.wait(t2)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_dp_step_rejects_bad_calls():
    """Refused with B2rlError before any launch, nothing changed: no graphs, n_new > capacity, a bad n_obs,
    wait_actions before any policy step; and the wide policy without a wide learner."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    with pytest.raises(L.B2rlError):
        _learner("sac", None, "wide")
    assert _learner("sac", "3xtf32").policy == "row"  # (the default: the row kernel measured faster, DESIGN §5)
    for dp, call in ((_learner("sac", None, graphs=False), lambda d: d.step_async(0, 8, 8)),
                     (_learner("td3", "3xtf32", cap=2500), lambda d: d.step_async(0, 2501, 8)),
                     (_learner("td3", None), lambda d: d.step_async(0, 8, -1)),
                     (_learner("td3", None), lambda d: d.step_async(0, 8, 2.5)),
                     (_learner("sac", None), lambda d: d.wait_actions())):
        torch.cuda.synchronize()
        before = _state(dp)
        with pytest.raises(L.B2rlError):
            call(dp)
        torch.cuda.synchronize()
        _assert_same(before, _state(dp), "refused call")
        assert dp._stage.seq == 0 and not dp._step_graphs


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_dp_step_matches_eager_protocol():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29537", str(REPO / "tests" / "dp_step_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=REPO, env=dict(os.environ))
    print(p.stdout[-3000:], p.stderr[-3000:])
    assert p.returncode == 0 and "DP_STEP_OK" in p.stdout
