"""TEST INFRASTRUCTURE ONLY — pure-torch oracle for the SAC/TD3 learner update.

A functional restatement (parameters live in plain ``dict[str, Tensor]``) of the
reference's update step, written so that every random draw (replay indices,
reparameterisation noise, TD3 smoothing noise) can be injected. The CUDA path
in ``sac_td3_cudagraphs_pytorch_b200`` is compared against this on identical
inputs; this file is never imported by the product.

Reference anchors (paths relative to /root/reference):
  * nets:     agents/nets.py:52-92 (Critic), :95-159 (Actor), :162-234 (TanhGaussActor),
              :34-49 (init), :13 (log-std bounds)
  * update:   agents/agent.py:146-170 (batched_qf / pi / alpha), :183-242 (update_qnets),
              :244-318 (update_actor), :320-331 (update_targ_nets)
  * cadence:  orchestrator.py:337-352
  * constants: tasks/defaults/sac.yml, tasks/defaults/td3.yml
  * Normal:   torch/distributions/normal.py (rsample = loc + eps*scale; log_prob)
  * Adam:     torch/optim/adam.py (_single_tensor_adam, both the host-scalar and the
              ``capturable`` device-scalar branch)

Parity: pinned against the reference's own code, see tests/golden/make_golden.py.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field, asdict
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

HID = 256  # agents/agent.py:56,101 hard-codes (256, 256)
LOG_STD_LO, LOG_STD_HI = -5.0, 2.0  # agents/nets.py:13
LN_EPS = 1e-5  # torch.nn.LayerNorm default, agents/nets.py:70,76

PARAM_NAMES = (
    "fc_stack.fc_block_1.fc.weight",
    "fc_stack.fc_block_1.fc.bias",
    "fc_stack.fc_block_1.ln.weight",
    "fc_stack.fc_block_1.ln.bias",
    "fc_stack.fc_block_2.fc.weight",
    "fc_stack.fc_block_2.fc.bias",
    "fc_stack.fc_block_2.ln.weight",
    "fc_stack.fc_block_2.ln.bias",
    "head.weight",
    "head.bias",
)
_LN_NAMES = tuple(n for n in PARAM_NAMES if ".ln." in n)


# --------------------------------------------------------------------------- hps
@dataclass
class OracleHps:
    """The keys Agent reads from the config (SURVEY.md §5 'Config / flags')."""

    prefer_td3_over_sac: bool = False
    layer_norm: bool = True
    batch_size: int = 256
    segment_len: int = 1
    gamma: float = 0.99
    polyak: float = 0.005
    actor_lr: float = 3e-4
    qnets_lr: float = 1e-3
    clip_norm: float = 0.0
    bcq_style_targ_mix: bool = False
    actor_update_delay: int = 2
    # SAC tail (sac.yml:44-48)
    crit_targ_update_freq: int = 1
    alpha_init: float = 0.2
    autotune: bool = True
    log_alpha_lr: float = 1e-3
    # TD3 tail (td3.yml:44-48)
    actor_noise_std: float = 0.1
    targ_actor_smoothing: bool = True
    td3_std: float = 0.2
    td3_c: float = 0.5
    # which torch Adam branch to mimic: False = host float64 bias corrections
    # (what the reference runs on CPU), True = device fp32 scalars (reference on GPU
    # with cudagraphs: agents/agent.py:118)
    adam_capturable: bool = False

    def to_dict(self):
        return asdict(self)


def sac_defaults(**kw) -> OracleHps:
    """tasks/defaults/sac.yml"""
    return OracleHps(prefer_td3_over_sac=False, qnets_lr=1e-3, bcq_style_targ_mix=False, **kw)


def td3_defaults(**kw) -> OracleHps:
    """tasks/defaults/td3.yml"""
    return OracleHps(prefer_td3_over_sac=True, qnets_lr=3e-4, bcq_style_targ_mix=True, **kw)


# -------------------------------------------------------------------------- nets
def init_mlp_params(in_dim: int, out_dim: int, *, layer_norm: bool, generator=None,
                    dtype=torch.float32) -> dict[str, torch.Tensor]:
    """Orthogonal(gain 1) weights, zero biases, LN ones/zeros (agents/nets.py:34-49)."""
    def ortho(o, i):
        w = torch.empty(o, i, dtype=torch.float32)
        torch.nn.init.orthogonal_(w, generator=generator)
        return w.to(dtype)

    p = {
        "fc_stack.fc_block_1.fc.weight": ortho(HID, in_dim),
        "fc_stack.fc_block_1.fc.bias": torch.zeros(HID, dtype=dtype),
        "fc_stack.fc_block_2.fc.weight": ortho(HID, HID),
        "fc_stack.fc_block_2.fc.bias": torch.zeros(HID, dtype=dtype),
        "head.weight": ortho(out_dim, HID),
        "head.bias": torch.zeros(out_dim, dtype=dtype),
    }
    if layer_norm:
        for blk in ("fc_block_1", "fc_block_2"):
            p[f"fc_stack.{blk}.ln.weight"] = torch.ones(HID, dtype=dtype)
            p[f"fc_stack.{blk}.ln.bias"] = torch.zeros(HID, dtype=dtype)
    return {k: p[k] for k in PARAM_NAMES if k in p}


def mlp_forward(p: dict[str, torch.Tensor], x: torch.Tensor, layer_norm: bool) -> torch.Tensor:
    """Linear -> [LayerNorm] -> ReLU, twice, then the head (agents/nets.py:66-92)."""
    for blk in ("fc_block_1", "fc_block_2"):
        x = F.linear(x, p[f"fc_stack.{blk}.fc.weight"], p[f"fc_stack.{blk}.fc.bias"])
        if layer_norm:
            x = F.layer_norm(x, (HID,), p[f"fc_stack.{blk}.ln.weight"],
                             p[f"fc_stack.{blk}.ln.bias"], LN_EPS)
        x = torch.relu(x)
    return F.linear(x, p["head.weight"], p["head.bias"])


def critic_forward(p, ob, ac, layer_norm):
    """agents/nets.py:88-92 — pack([ob, ac]) then the MLP, output [B,1]."""
    return mlp_forward(p, torch.cat([ob, ac], dim=-1), layer_norm)


def normal_log_prob(value, loc, scale):
    """torch.distributions.Normal.log_prob, expression order preserved."""
    var = scale ** 2
    log_scale = scale.log()
    return -((value - loc) ** 2) / (2 * var) - log_scale - math.log(math.sqrt(2 * math.pi))


# ----------------------------------------------------------------- portable RNG
_PHILOX_M0 = np.uint64(0xD2511F53)
_PHILOX_M1 = np.uint64(0xCD9E8D57)
_PHILOX_W0 = np.uint32(0x9E3779B9)
_PHILOX_W1 = np.uint32(0xBB67AE85)


def philox4x32_10(counter: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox-4x32-10 (Salmon et al. 2011). counter [...,4] u32, key [...,2] u32 -> [...,4] u32.

    The CUDA kernels implement the same function (csrc/rng.cuh); integer math, so
    the two agree bit for bit.
    """
    c = np.array(counter, dtype=np.uint32, copy=True)
    k = np.array(np.broadcast_to(np.asarray(key, dtype=np.uint32), c.shape[:-1] + (2,)), copy=True)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = _PHILOX_M0 * c[..., 0].astype(np.uint64)
            p1 = _PHILOX_M1 * c[..., 2].astype(np.uint64)
            hi0 = (p0 >> np.uint64(32)).astype(np.uint32)
            lo0 = p0.astype(np.uint32)
            hi1 = (p1 >> np.uint64(32)).astype(np.uint32)
            lo1 = p1.astype(np.uint32)
            c = np.stack([hi1 ^ c[..., 1] ^ k[..., 0], lo1, hi0 ^ c[..., 3] ^ k[..., 1], lo0], axis=-1)
            k = np.stack([k[..., 0] + _PHILOX_W0, k[..., 1] + _PHILOX_W1], axis=-1)
    return c


# stream ids shared with csrc/rng.cuh
STREAM_INDEX, STREAM_CRITIC_EPS, STREAM_ACTOR_EPS, STREAM_ALPHA_EPS = 0, 1, 2, 3


def _ctr(a, b, step, stream_agent):
    a = np.asarray(a, dtype=np.uint32)
    out = np.zeros(a.shape + (4,), dtype=np.uint32)
    out[..., 0] = a
    out[..., 1] = np.uint32(b) if np.isscalar(b) else np.asarray(b, dtype=np.uint32)
    out[..., 2] = np.uint32(step & 0xFFFFFFFF)
    out[..., 3] = np.uint32(stream_agent)
    return out


def philox_randint(seed: int, step: int, n: int, batch: int, agent: int = 0) -> np.ndarray:
    """Replay indices as csrc/replay.cu draws them: idx = (r0 * n) >> 32, one Philox block per row."""
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    r = philox4x32_10(_ctr(np.arange(batch), 0, step, (agent << 2) | STREAM_INDEX), key)
    return ((r[..., 0].astype(np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def philox_normal_pairs(seed: int, step: int, stream: int, batch: int, dim: int,
                        agent: int = 0) -> np.ndarray:
    """N(0,1) noise [batch, dim] as the kernels draw it (Box-Muller on Philox words).

    Float transcendental rounding differs between libm and the GPU, so this matches
    the device to ~1e-6, not bit for bit; parity tests read the noise back from the
    kernel instead (``eps_out``)."""
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    nblk = (dim + 3) // 4
    b = np.arange(batch)[:, None].repeat(nblk, 1)
    q = np.arange(nblk)[None, :].repeat(batch, 0)
    r = philox4x32_10(_ctr(b, q, step, (agent << 2) | stream), key)  # [B, nblk, 4]
    u = r.astype(np.float64)
    out = np.empty((batch, nblk, 4), dtype=np.float32)
    for h in range(2):
        u1 = ((u[..., 2 * h] + 1.0) * 2.0 ** -32).astype(np.float32)
        u2 = (u[..., 2 * h + 1] * 2.0 ** -32).astype(np.float32)
        rad = np.sqrt(np.float32(-2.0) * np.log(u1)).astype(np.float32)
        ang = np.float32(2.0 * math.pi) * u2
        out[..., 2 * h] = rad * np.cos(ang)
        out[..., 2 * h + 1] = rad * np.sin(ang)
    return out.reshape(batch, nblk * 4)[:, :dim]


# -------------------------------------------------------------- synthetic data
def make_synthetic_transitions(n: int, ob_dim: int, ac_dim: int, min_ac, max_ac, seed: int = 1234,
                               device="cpu") -> dict[str, torch.Tensor]:
    """SURVEY.md §8(d): obs~N(0,1), next=obs+0.1N(0,1), act~U(min,max), rew~N(0,1), done~Bern(0.01)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    lo = torch.as_tensor(min_ac, dtype=torch.float32)
    hi = torch.as_tensor(max_ac, dtype=torch.float32)
    obs = torch.randn(n, ob_dim, generator=g)
    nxt = obs + 0.1 * torch.randn(n, ob_dim, generator=g)
    act = lo + (hi - lo) * torch.rand(n, ac_dim, generator=g)
    rew = torch.randn(n, 1, generator=g)
    done = torch.rand(n, 1, generator=g) < 0.01
    td = {
        "observations": obs, "next_observations": nxt, "actions": act, "rewards": rew,
        "terminations": done, "dones": done.clone(),
    }
    return {k: v.to(device) for k, v in td.items()}


# ------------------------------------------------------------------------ Adam
class _Adam:
    """torch.optim.Adam(betas=(0.9,0.999), eps=1e-8, wd=0) restated for one param group.

    ``capturable=False`` follows torch/optim/adam.py:528-550 (bias corrections in host
    float64, ``addcdiv_(m, denom, value=-step_size)``); ``capturable=True`` follows
    :478-527 (fp32 device scalars, ``denom = sqrt(v)/(bc2_sqrt*(-ss)) + eps/(-ss)``;
    ``p += m/denom``). In the capturable branch the step count is a float32 tensor, so the
    bias corrections are fp32 whatever the dtype of the parameters: a float64 oracle is
    float64 in its optimizer only with ``capturable=False``. Checked against
    torch.optim.Adam in tests/test_gpu_optimizer.py (``test_oracle_adam_matches_torch``:
    both branches, the capturable one on the GPU).
    """

    def __init__(self, params, lr, capturable=False, b1=0.9, b2=0.999, eps=1e-8):
        self.params = list(params)
        self.lr, self.b1, self.b2, self.eps, self.capturable = lr, b1, b2, eps, capturable
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.t = 0

    def zero_grad(self):
        for p in self.params:
            p.grad = None

    @torch.no_grad()
    def step(self):
        self.t += 1
        for p, m, v in zip(self.params, self.m, self.v):
            g = p.grad
            if g is None:
                continue
            m.lerp_(g, 1 - self.b1)
            v.mul_(self.b2).addcmul_(g, g, value=1 - self.b2)
            if self.capturable:
                step = torch.tensor(float(self.t), dtype=torch.float32, device=p.device)
                bc1 = 1 - self.b1 ** step
                bc2 = 1 - self.b2 ** step
                ss_neg = (self.lr / bc1).neg()
                denom = (v.sqrt() / (bc2.sqrt() * ss_neg)).add_(self.eps / ss_neg)
                p.addcdiv_(m, denom.to(p.dtype))
            else:
                bc1 = 1 - self.b1 ** self.t
                bc2 = 1 - self.b2 ** self.t
                denom = (v.sqrt() / (bc2 ** 0.5)).add_(self.eps)
                p.addcdiv_(m, denom, value=-(self.lr / bc1))


# ----------------------------------------------------------------------- agent
class OracleAgent:
    """Learner state + the three update functions of agents/agent.py, functionally.

    ``actor`` / ``actor_target``: dict name -> tensor. ``qnet`` / ``qnet_target``: dict
    name -> tensor stacked on a leading dim of 2, evaluated with ``torch.vmap`` exactly
    like ``TensorDict.from_modules(q1, q2)`` + ``torch.vmap(batched_qf)`` in the
    reference (agents/agent.py:106, :208, :230), so the GEMMs lower to the same bmm.
    """

    def __init__(self, ob_dim: int, ac_dim: int, min_ac, max_ac, hps: OracleHps,
                 device="cpu", dtype=torch.float32, seed: int = 0,
                 actor_init: Optional[dict] = None, qnet_init: Optional[list[dict]] = None,
                 torch_adam: bool = False):
        self.ob_dim, self.ac_dim, self.hps = ob_dim, ac_dim, hps
        self.device, self.dtype = torch.device(device), dtype
        self.td3 = bool(hps.prefer_td3_over_sac)
        self.min_ac = torch.as_tensor(np.asarray(min_ac), dtype=dtype, device=self.device)
        self.max_ac = torch.as_tensor(np.asarray(max_ac), dtype=dtype, device=self.device)
        self.action_scale = (self.max_ac - self.min_ac) / 2.0  # agents/nets.py:200-204
        self.action_bias = (self.max_ac + self.min_ac) / 2.0
        assert hps.segment_len <= hps.batch_size  # agents/agent.py:47

        g = torch.Generator().manual_seed(seed)
        a_out = ac_dim if self.td3 else 2 * ac_dim
        if actor_init is None:
            actor_init = init_mlp_params(ob_dim, a_out, layer_norm=hps.layer_norm, generator=g)
        if qnet_init is None:
            qnet_init = [init_mlp_params(ob_dim + ac_dim, 1, layer_norm=hps.layer_norm, generator=g)
                         for _ in range(2)]

        def leaf(t):
            return t.detach().to(self.device, dtype).clone().requires_grad_(True)

        self.actor = {k: leaf(v) for k, v in actor_init.items()}
        self.actor_target = {k: v.detach().clone() for k, v in self.actor.items()}
        self.qnet = {k: leaf(torch.stack([qnet_init[0][k], qnet_init[1][k]])) for k in qnet_init[0]}
        self.qnet_target = {k: v.detach().clone() for k, v in self.qnet.items()}

        cap = hps.adam_capturable
        if torch_adam:  # the real torch.optim.Adam, as agents/agent.py:115-139 (capturable on the GPU)
            _mk = lambda ps, lr: torch.optim.Adam(list(ps), lr=lr, capturable=self.device.type == "cuda")
        else:
            _mk = lambda ps, lr: _Adam(ps, lr, cap)
        self.q_optimizer = _mk(self.qnet.values(), hps.qnets_lr)
        self.actor_optimizer = _mk(self.actor.values(), hps.actor_lr)
        if not self.td3:
            self.log_alpha = torch.tensor(hps.alpha_init, dtype=dtype, device=self.device).log()
            if hps.autotune:
                self.log_alpha.requires_grad_(True)
                self.targ_ent = -ac_dim  # agents/agent.py:134
                self.alpha_optimizer = _mk([self.log_alpha], hps.log_alpha_lr)
        self.qnet_updates_so_far = 0
        self.actor_updates_so_far = 0

    # -- pieces ------------------------------------------------------------
    @property
    def alpha(self):
        return None if self.td3 else self.log_alpha.exp()

    def pi(self, p, ob):
        """TD3 deterministic policy, agents/nets.py:143-147."""
        return torch.tanh(mlp_forward(p, ob, self.hps.layer_norm)) * self.action_scale + self.action_bias

    def get_action(self, p, ob, eps):
        """SAC tanh-Gaussian sample / log-prob / mode, agents/nets.py:206-234, noise injected."""
        mean, ls = mlp_forward(p, ob, self.hps.layer_norm).chunk(2, dim=-1)
        ls = torch.tanh(ls)
        ls = LOG_STD_LO + 0.5 * (LOG_STD_HI - LOG_STD_LO) * (ls + 1)
        std = ls.exp()
        x_t = mean + eps * std  # Normal.rsample
        y_t = torch.tanh(x_t)
        action = y_t * self.action_scale + self.action_bias
        log_prob = normal_log_prob(x_t, mean, std)
        log_prob = log_prob - torch.log(self.action_scale * (1 - y_t.pow(2)) + 1e-6)
        log_prob = log_prob.sum(1, keepdim=True)
        mode = torch.tanh(mean) * self.action_scale + self.action_bias
        return action, log_prob, mode

    def qf(self, stacked, ob, ac):
        ln = self.hps.layer_norm
        return torch.vmap(lambda p, o, a: critic_forward(p, o, a, ln), (0, None, None))(stacked, ob, ac)

    def _eps(self, eps, like):
        if eps is None:
            return torch.randn_like(like)
        return torch.as_tensor(eps, dtype=self.dtype, device=self.device)

    # -- agents/agent.py:183-242 ---------------------------------------------
    def update_qnets(self, batch, eps=None):
        h = self.hps
        self.q_optimizer.zero_grad()
        with torch.no_grad():
            nob = batch["next_observations"]
            if self.td3:
                next_logpi = None
                pi_next = self.pi(self.actor_target, nob)
                if h.targ_actor_smoothing:
                    n_ = self._eps(eps, batch["actions"]) * h.td3_std
                    n_ = n_.clamp(-h.td3_c, h.td3_c)
                    next_action = (pi_next + n_).clamp(self.min_ac, self.max_ac)
                else:
                    next_action = pi_next
            else:
                next_action, next_logpi, _ = self.get_action(self.actor, nob, self._eps(eps, batch["actions"]))
            qf_next = self.qf(self.qnet_target, nob, next_action)
            qf_min = qf_next.min(0).values
            if h.bcq_style_targ_mix:
                q_prime = 0.75 * qf_min + 0.25 * qf_next.max(0).values
            else:
                q_prime = qf_min
            if not self.td3:
                q_prime = q_prime - self.alpha * next_logpi
            targ_q = batch["rewards"].flatten() + (~batch["dones"].flatten()).to(self.dtype) \
                * h.gamma * q_prime.view(-1)
        ln = h.layer_norm

        def per_critic_mse(p, ob, ac, y):  # batched_qf with next_q_value given (:146-157)
            vals = critic_forward(p, ob, ac, ln)
            return F.mse_loss(vals.view(-1), y), vals.view(-1)

        per_critic, q = torch.vmap(per_critic_mse, (0, None, None, None))(
            self.qnet, batch["observations"], batch["actions"], targ_q)
        qf_loss = per_critic.sum(0)
        qf_loss.backward()
        self.q_optimizer.step()
        # NB: the reference bumps qnet_updates_so_far in orchestrator.py:342, not here
        return {"loss/qf_loss": qf_loss.detach(), "_targ_q": targ_q, "_q": q.detach()}

    # -- agents/agent.py:244-318 ---------------------------------------------
    def update_actor(self, batch, eps=None, eps_alpha=None):
        h = self.hps
        ob = batch["observations"]
        self.actor_optimizer.zero_grad()
        qdet = {k: v.detach() for k, v in self.qnet.items()}
        if self.td3:
            a = self.pi(self.actor, ob)
            actor_loss = -self.qf(qdet, ob, a)[0]
        else:
            a, logpi, _ = self.get_action(self.actor, ob, self._eps(eps, batch["actions"]))
            actor_loss = self.alpha.detach() * logpi - self.qf(qdet, ob, a).min(0).values
        actor_loss = actor_loss.mean()
        actor_loss.backward()
        if h.clip_norm > 0:
            torch.nn.utils.clip_grad_norm_(list(self.actor.values()), h.clip_norm)
        self.actor_optimizer.step()
        out = {"loss/actor_loss": actor_loss.detach()}
        if self.td3:
            return out
        if h.autotune:
            self.alpha_optimizer.zero_grad()
            with torch.no_grad():
                _, logpi2, _ = self.get_action(self.actor, ob, self._eps(eps_alpha, batch["actions"]))
            alpha_loss = (self.alpha * (-logpi2 - self.targ_ent).detach()).mean()
            alpha_loss.backward()
            self.alpha_optimizer.step()
            out["loss/alpha_loss"] = alpha_loss.detach()
        out["vitals/alpha"] = self.alpha.detach()
        return out

    # -- agents/agent.py:320-331 ---------------------------------------------
    @torch.no_grad()
    def update_targ_nets(self):
        h = self.hps
        if self.td3 or (self.qnet_updates_so_far % h.crit_targ_update_freq == 0):
            for k, t in self.qnet_target.items():
                t.lerp_(self.qnet[k].detach(), h.polyak)
            if self.td3:
                for k, t in self.actor_target.items():
                    t.lerp_(self.actor[k].detach(), h.polyak)

    # -- orchestrator.py:337-352 --------------------------------------------
    def iteration(self, i: int, batch, eps_q=None, eps_pi=None, eps_alpha=None):
        """One learner iteration in the reference cadence. ``eps_pi`` / ``eps_alpha`` are lists
        (one entry per delayed actor update)."""
        logs = dict(self.update_qnets(batch, eps_q))
        self.qnet_updates_so_far += 1  # orchestrator.py:342
        if i % (self.hps.actor_update_delay + 1) == 0:
            for j in range(self.hps.actor_update_delay):
                e1 = None if eps_pi is None else eps_pi[j]
                e2 = None if eps_alpha is None else eps_alpha[j]
                logs.update(self.update_actor(batch, e1, e2))
                self.actor_updates_so_far += 1  # orchestrator.py:349
        self.update_targ_nets()
        return logs

    # -- helpers for tests ------------------------------------------------------
    def critic_state(self, k: int, target=False):
        src = self.qnet_target if target else self.qnet
        return {n: v[k].detach().clone() for n, v in src.items()}

    def actor_state(self, target=False):
        src = self.actor_target if target else self.actor
        return {n: v.detach().clone() for n, v in src.items()}

    def sample_batch(self, storage: dict[str, torch.Tensor], idx) -> dict[str, torch.Tensor]:
        """torchrl LazyTensorStorage + RandomSampler semantics: per-key ``storage[key][idx]``."""
        idx = torch.as_tensor(idx, dtype=torch.long, device=self.device)
        out = {k: v[idx] for k, v in storage.items()}
        out["index"] = idx
        return out
