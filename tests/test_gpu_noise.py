"""The device-drawn noise against its numpy twin, and the behaviour policy against a float64 forward pass.

Every N(0,1) the kernels draw themselves is box_muller4(philox_block(...)) of csrc/rng.cuh, keyed on
(seed; row, Philox block, 32-bit step, global agent id << 2 | stream). oracle.philox_normal_pairs is the same
function in numpy. The tests below read the draws back (eps_out / eps2_out, the wide actor's save buffer, the
behaviour policy's actions) and compare them with the twin, so a wrong key, step counter, row <-> block mapping or
agent id fails here even where graph == eager, stacked == single and sharded == whole all still hold.

Error model of a draw (z = r cos(theta), r = sqrt(-2 ln u1), theta = 2 pi u2), element by element:
  - ln u1: __logf has an absolute error <= 2^-21.41 on [0.5, 2] and <= 3 ulp elsewhere (CUDA C Programming Guide,
    intrinsic functions); the device rounds u1 = ((float)w + 1) * 2^-32 twice, the twin once, so u1 may differ by one
    ulp: + 2^-23 in ln u1.
  - r: r^2 = -2 ln u1 moves by 2 d(ln u1), so |dr| <= min(2 d / r, sqrt(2 d)). Where u1 is within 2^-16 of 1 the radius is
    the square root of a tiny number and this term reaches ~1e-3; those elements are counted and reported apart.
  - theta: __sincosf is the MUFU approximation after a multiply by 1/(2 pi): <= 2^-21.41 + 2 pi 2^-24 absolute, times r.
  - fp32 rounding of sqrt, of the products and of the twin's own result: 2^-22 (|z| + r).
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions, philox4x32_10, philox_normal_pairs
from oracle.sac_td3_oracle import STREAM_ACTOR_EPS, STREAM_ALPHA_EPS, STREAM_CRITIC_EPS, mlp_forward

M64 = (1 << 64) - 1
SEED_HI = 0x9E3779B97F4A7C15  # a key with a non-zero high word (the Philox key is the whole 64-bit seed)
EPS_LOG = 2.0 ** -21.41
EPS_TRIG = 2.0 ** -21.41 + 2.0 * math.pi * 2.0 ** -24
U1_EDGE = 1.0 - 2.0 ** -16
R_MAX = math.sqrt(-2.0 * math.log(2.0 ** -32))  # the largest radius: u1 = 2^-32


# ---------------------------------------------------------------------------------------------------- the twin
def _words(seed, step, stream, rows, blocks, agent):
    """Philox words [len(rows), len(blocks), 4] of counter (row, block, step & 0xFFFFFFFF, agent << 2 | stream)."""
    c = np.zeros((len(rows), len(blocks), 4), dtype=np.uint32)
    c[..., 0] = np.asarray(rows, dtype=np.uint32)[:, None]
    c[..., 1] = np.asarray(blocks, dtype=np.uint32)[None, :]
    c[..., 2] = np.uint32(step & 0xFFFFFFFF)
    c[..., 3] = np.uint32(((agent << 2) | stream) & 0xFFFFFFFF)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32)
    return philox4x32_10(c, key)


def twin(seed, step, stream, B, A, agent):
    """(z, u1): the twin's draws [B, A] (oracle.philox_normal_pairs) and the fp32 u1 each element's radius came from."""
    z = philox_normal_pairs(seed & M64, step & 0xFFFFFFFF, stream, B, A, agent)
    nblk = (A + 3) // 4
    w = _words(seed & M64, step, stream, np.arange(B), np.arange(nblk), agent).astype(np.float64)
    u1 = ((w[..., [0, 0, 2, 2]] + 1.0) * 2.0 ** -32).astype(np.float32).astype(np.float64)
    return z, u1.reshape(B, 4 * nblk)[:, :A]


def noise_tol(u1, z):
    """Per-element bound |device - twin| of the module docstring's error model."""
    L = np.log(u1)
    r = np.sqrt(-2.0 * L)
    d = np.where(u1 >= 0.5, EPS_LOG, 3 * 2.0 ** -23 * np.abs(L)) + 2.0 ** -23
    with np.errstate(divide="ignore"):
        dr = np.minimum(np.where(r > 0, 2 * d / np.maximum(r, 1e-30), np.inf), np.sqrt(2 * d))
    return dr + r * EPS_TRIG + 2.0 ** -22 * (np.abs(z) + r)


class Worst:
    """The worst deviations of many draws, reported once per test: bulk |dz| (u1 <= 1 - 2^-16), the elements with
    u1 > 1 - 2^-16 (count and worst |dz|) and the worst ratio to the element-wise bound."""

    def __init__(self):
        self.rows = {}

    def add(self, key, bulk, n_edge, edge, ratio):
        b0, n0, e0, r0 = self.rows.get(key, (0.0, 0, 0.0, 0.0))
        self.rows[key] = (max(b0, bulk), n0 + n_edge, max(e0, edge), max(r0, ratio))

    def report(self):
        for key, (b, n, e, r) in self.rows.items():
            print(f"{key}: worst |dz| {b:.2e}; {n} draws with u1 > 1-2^-16, worst |dz| {e:.2e}; worst dev/bound {r:.3f}")


def check_noise(what, got, seed, step, stream, agent, worst=None, key=None):
    """got [B, A] (device) against the twin, element by element (noise_tol); returns the bound for callers that
    propagate it. worst / key: accumulate the deviations under key instead of printing them."""
    got = torch.as_tensor(got).detach().cpu().double().numpy()
    B, A = got.shape
    z, u1 = twin(seed, step, stream, B, A, agent)
    tol = noise_tol(u1, z)
    assert np.isfinite(got).all(), f"{what}: non-finite draws at {np.argwhere(~np.isfinite(got))[:4].tolist()}"
    dev = np.abs(got - z)
    edge = u1 > U1_EDGE
    stats = (float(dev[~edge].max()) if (~edge).any() else 0.0, int(edge.sum()), float(dev[edge].max()) if edge.any() else 0.0,
             float((dev / tol).max()))
    if worst is None:
        one = Worst()
        one.add(what, *stats)
        one.report()
    else:
        worst.add(key or what, *stats)
    bad = np.argwhere(dev > tol)
    assert bad.size == 0, f"{what}: |device - twin| above the bound at (row, dim, device, twin, bound) " + str(
        [(int(i), int(j), got[i, j], float(z[i, j]), float(tol[i, j])) for i, j in bad[:4]])
    return tol


# ---------------------------------------------------------------------------------------------------- fixtures
def _hps(kind, **over):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    if kind == "sac":
        return sac_hps(**over)
    return td3_hps(targ_actor_smoothing=(kind == "td3"), **over)


def _rows(n, ob, A, lo, hi, seed):
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows, row_format
    td = make_synthetic_transitions(n, ob, A, lo, hi, seed=seed)
    return pack_rows({k: v.cuda() for k, v in td.items()}, row_format(ob, A))


_AGENTS = {}


def _agent(kind, A, ob=11, seed=SEED_HI, layer_norm=True, lo=None, hi=None, cache=True):
    """An Agent with bounds [lo, hi] (default [-1, 1]); cached per configuration for the whole module unless cache=False
    (agent_id and counters are set by each test)."""
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    lo = [-1.0] * A if lo is None else list(lo)
    hi = [1.0] * A if hi is None else list(hi)
    key = (kind, A, ob, seed, layer_norm, tuple(lo), tuple(hi))
    if key in _AGENTS:
        return _AGENTS[key]
    ag = Agent({"ob_shape": (ob,), "ac_shape": (A,)}, np.array(lo, np.float32), np.array(hi, np.float32),
               torch.device("cuda"), _hps(kind, layer_norm=layer_norm), rb=None, seed=seed)
    if cache:
        _AGENTS[key] = ag
    return ag


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


# the step counters the noise is keyed on: 0, both sides of bit 31, the 32-bit wrap, and far above it
STEPS = (0, 5, (1 << 31) - 1, 1 << 31, (1 << 32) - 1, (1 << 32) + 3, (1 << 45) + 12345)
AGENT_IDS = (0, 3, (1 << 30) - 1)


# ---------------------------------------------------------------------------------------------------- 1. row path
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 7, 9, 256, 1000])
@pytest.mark.parametrize("A", [1, 3, 4, 5, 8, 17])
def test_row_path_noise_matches_the_twin(A, B):
    """The fused critic, actor and temperature kernels' own draws == the twin, with the counter each one reads:
    the critic CTR_Q, the actor CTR_PI, the temperature CTR_PI after the actor step's weight-gradient launch advanced it.
    TD3 without target smoothing and TD3's actor step draw nothing (eps_out stays untouched)."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ob = 11
    rows = _rows(B, ob, A, [-1.0] * A, [1.0] * A, seed=100 + A)
    worst = Worst()
    for kind in ("sac", "td3", "td3_nosmooth"):
        ag = _agent(kind, A)
        for i, aid in enumerate(AGENT_IDS):
            ag.agent_id = aid
            for c in (STEPS[i::2] if B > 256 else STEPS):
                # ---- critic step: next-action sample (SAC) / target smoothing (TD3)
                ag.counters[L.CTR_Q] = c
                eo = _nan(B, A)
                ag.update_qnets(rows, eps_out=eo)
                torch.cuda.synchronize()
                assert int(ag.counters[L.CTR_Q]) == c + 1
                tag = f"{kind} critic A={A} B={B} agent={aid} step={c:#x}"
                if kind == "td3_nosmooth":
                    assert torch.isnan(eo).all(), tag + ": drew noise without target smoothing"
                else:
                    check_noise(tag, eo, SEED_HI, c, STREAM_CRITIC_EPS, aid, worst, f"{kind} critic A={A} B={B}")
                # ---- actor step (+ SAC temperature step)
                ag.counters[L.CTR_PI] = c
                eo, eo2 = _nan(B, A), _nan(B, A)
                ag.update_actor(rows, eps_out=eo, eps2_out=eo2)
                torch.cuda.synchronize()
                assert int(ag.counters[L.CTR_PI]) == c + 1
                tag = f"{kind} actor A={A} B={B} agent={aid} step={c:#x}"
                if kind == "sac":
                    check_noise(tag, eo, SEED_HI, c, STREAM_ACTOR_EPS, aid, worst, f"sac actor A={A} B={B}")
                    check_noise(f"sac alpha A={A} B={B} agent={aid} step={c + 1:#x}", eo2, SEED_HI, c + 1,
                                STREAM_ALPHA_EPS, aid, worst, f"sac alpha A={A} B={B}")
                else:
                    assert torch.isnan(eo).all() and torch.isnan(eo2).all(), tag + ": TD3's actor step drew noise"
    worst.report()


def _population(ids, kind, A, B, seed, wide=None):
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, 11, A, [-1.0] * A, [1.0] * A, _hps(kind, batch_size=B), "cuda", seed=seed, rb_capacity=64,
                     use_graphs=False, wide=wide)
    for g in range(len(ids)):
        pop.rows[g].copy_(_rows(B, 11, A, [-1.0] * A, [1.0] * A, seed=200 + g))
    return pop


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sac", "td3"])
def test_stacked_launch_keys_agent_g_on_base_plus_g(kind):
    """Agents stacked in grid y with agent_base = 5: agent g draws with global id 5 + g and its own counters."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ids, A, B, seed = [5, 6, 7], 5, 19, 0xFFFFFFFF00000001
    pop = _population(ids, kind, A, B, seed)
    lib, st = pop._lib, torch.cuda.current_stream().cuda_stream
    steps = [3, (1 << 32) + 17, (1 << 31) + 1]
    for g, c in enumerate(steps):
        pop.counters[g, L.CTR_Q] = c
        pop.counters[g, L.CTR_PI] = c + 100
    eo, eo_pi, eo2 = _nan(3, B, A), _nan(3, B, A), _nan(3, B, A)
    args = L.UpdateArgs.from_buffer_copy(pop.args)
    args.eps_out, args.eps2_out = eo.data_ptr(), eo2.data_ptr()
    crit = lib.b2rl_critic_update_td3 if kind == "td3" else lib.b2rl_critic_update_sac
    L.check(crit(C.byref(args), st), "critic_update")
    args.eps_out = eo_pi.data_ptr()
    L.check((lib.b2rl_actor_update_td3 if kind == "td3" else lib.b2rl_actor_update_sac)(C.byref(args), st), "actor_update")
    if kind == "sac":
        L.check(lib.b2rl_alpha_update(C.byref(args), 1e-3, st), "alpha_update")
    torch.cuda.synchronize()
    for g, c in enumerate(steps):
        assert int(pop.counters[g, L.CTR_Q]) == c + 1 and int(pop.counters[g, L.CTR_PI]) == c + 101
        check_noise(f"stacked {kind} critic g={g} agent={ids[g]}", eo[g], seed, c, STREAM_CRITIC_EPS, ids[g])
        if kind == "sac":
            check_noise(f"stacked sac actor g={g}", eo_pi[g], seed, c + 100, STREAM_ACTOR_EPS, ids[g])
            check_noise(f"stacked sac alpha g={g}", eo2[g], seed, c + 101, STREAM_ALPHA_EPS, ids[g])
        else:
            assert torch.isnan(eo_pi[g]).all() and torch.isnan(eo2[g]).all()


# ---------------------------------------------------------------------------------------------------- 2. wide path
@pytest.mark.gpu
@pytest.mark.parametrize("A", [3, 17])
@pytest.mark.parametrize("kind", ["sac", "td3"])
def test_wide_path_noise_matches_the_twin(kind, A):
    """The tensor-core path's policy head (wide.cu) keys its draws like the row path: the critic step's next-action noise
    (eps_out) on CTR_Q and stream 1, the SAC actor's sample (save[:, 0, :]) on CTR_PI and stream 2, per global agent id.
    B = 200 is ragged against the 128-row tiles."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ids, B, seed = [5, 6, 7], 200, SEED_HI
    pop = _population(ids, kind, A, B, seed, wide="3xtf32")
    steps = [11, (1 << 32) + 2, (1 << 31) - 1]
    for g, c in enumerate(steps):
        pop.counters[g, L.CTR_Q] = c
        pop.counters[g, L.CTR_PI] = c ^ (1 << 33)
    eo = _nan(3, B, A)
    pop.wide_q.update_qnets(pop.rows, eps_out=eo)
    pop.wide_pi.update_actor(pop.rows)
    torch.cuda.synchronize()
    save = pop.wide_pi.save.view(3, B, 4, A)
    for g, c in enumerate(steps):
        assert int(pop.counters[g, L.CTR_Q]) == c + 1 and int(pop.counters[g, L.CTR_PI]) == (c ^ (1 << 33)) + 1
        check_noise(f"wide {kind} critic A={A} g={g}", eo[g], seed, c, STREAM_CRITIC_EPS, ids[g])
        if kind == "sac":
            check_noise(f"wide sac actor A={A} g={g}", save[g, :, 0, :], seed, c ^ (1 << 33), STREAM_ACTOR_EPS, ids[g])


# ---------------------------------------------------------------------------------------------------- 3. Box-Muller edges
# Counters found with the twin (a search over 2^24 steps each). (name, seed, stream, agent, row, block, step, pair,
# Philox word u1 came from, word u2 came from); pair h uses words (2h, 2h + 1), i.e. action dims 4 * block + 2h, + 1.
CRITIC_EDGES = [
    ("u1 = 1 (w >= 2^32 - 128: z = 0)", 0, STREAM_CRITIC_EPS, 0, 0, 0, 10000704, 0, 4294967208, 3663900757),
    ("u1 = 1 - 2^-24", 0, STREAM_CRITIC_EPS, 0, 0, 0, 1670983, 1, 4294966950, 3377869173),
    ("u1 = 1 - 2^-24, second", 0, STREAM_CRITIC_EPS, 0, 0, 0, 9698461, 0, 4294967124, 1003552296),
    ("u2 = 1 (angle 2 pi)", 0, STREAM_CRITIC_EPS, 0, 0, 0, 4847881, 0, 3136642196, 4294967197),
    ("tail: u1 = 67 * 2^-32, |z| ~ 6", 0, STREAM_CRITIC_EPS, 0, 0, 0, 1054365, 0, 66, 252758476),
]
# the behaviour policy: key ~seed, stream 2, steps >= 2^31 (what draw = ~0 makes of a critic counter)
PREDICT_EDGES = [
    ("u1 = 1 - 2^-24", M64, STREAM_ACTOR_EPS, 0, 0, 0, 2155469975, 0, 4294966948, 1139550038),
    ("u2 = 1 (angle 2 pi)", M64, STREAM_ACTOR_EPS, 0, 0, 0, 2158184544, 1, 4026783040, 4294967294),
    ("tail: u1 = 131 * 2^-32", M64, STREAM_ACTOR_EPS, 0, 0, 0, 2150740169, 1, 130, 3336056981),
]
EDGES = CRITIC_EDGES + PREDICT_EDGES


@pytest.mark.parametrize("edge", EDGES, ids=[f"{e[2]}-{e[0]}" for e in EDGES])
def test_edge_counters_give_the_claimed_philox_words(edge):
    """CPU only: the hard-coded counters produce the Philox words that make them edge cases, and the twin's draws there
    are finite and within the largest radius."""
    name, seed, stream, agent, row, blk, step, h, w1, w2 = edge
    r = _words(seed, step, stream, [row], [blk], agent)[0, 0]
    assert (int(r[2 * h]), int(r[2 * h + 1])) == (w1, w2), name
    u1 = np.float32((w1 + 1.0) * 2.0 ** -32)
    u2 = np.float32(w2 * 2.0 ** -32)
    if w1 >= 2 ** 32 - 128:
        assert u1 == np.float32(1.0)
    elif w1 >= 2 ** 32 - 384:
        assert u1 == np.float32(1.0 - 2.0 ** -24)
    if w2 >= 2 ** 32 - 128:
        assert u2 == np.float32(1.0)
    z, _ = twin(seed, step, stream, 1, 4 * blk + 4, agent)
    pair = z[0, 4 * blk + 2 * h: 4 * blk + 2 * h + 2]
    assert np.isfinite(pair).all() and (np.abs(pair) <= R_MAX).all()
    if w1 < 2 ** 20:
        assert np.hypot(*pair) > 5.0, name
    print(f"{name}: step {step} words ({w1:#x}, {w2:#x}) -> twin z = {pair.tolist()}")


@pytest.mark.gpu
@pytest.mark.parametrize("edge", CRITIC_EDGES, ids=[e[0] for e in CRITIC_EDGES])
def test_critic_draws_at_box_muller_edges(edge):
    """The critic kernel driven onto each edge counter: finite draws within the bound, equal to the twin, and the step
    they feed stays finite (a NaN here would poison the agent's parameters for good)."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    name, seed, stream, agent, row, blk, step, h, _, _ = edge
    A, B = 8, 8
    ag = _agent("sac", A, seed=seed)
    ag.agent_id = agent
    ag.counters[L.CTR_Q] = step
    eo = _nan(B, A)
    out = ag.update_qnets(_rows(B, 11, A, [-1.0] * A, [1.0] * A, seed=5), eps_out=eo)
    torch.cuda.synchronize()
    check_noise(f"edge critic {name}", eo, seed, step, stream, agent)
    d = 4 * blk + 2 * h
    pair = eo[row, d:d + 2].double().cpu()
    print(f"edge critic {name}: device z = {pair.tolist()}")
    assert (pair.abs() <= R_MAX).all()
    assert math.isfinite(float(out["loss/qf_loss"])) and torch.isfinite(ag.arena.flat).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sac", "td3"])
@pytest.mark.parametrize("edge", PREDICT_EDGES, ids=[e[0] for e in PREDICT_EDGES])
def test_behaviour_policy_at_box_muller_edges(edge, kind):
    """predict_kernel driven onto each edge counter, as a host-counted draw and as draw = ~0 on the critic counter:
    finite actions inside the bounds; for TD3 the recovered noise (a - mode) / (scale std) equals the twin."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    name, key, stream, agent, row, blk, step, h, _, _ = edge
    seed = key ^ M64
    A, n = 4 * blk + 4, 8
    ag = _agent(kind, A, seed=seed)
    ag.agent_id = agent
    obs = torch.randn(n, 11, generator=torch.Generator().manual_seed(9)).cuda()
    a0 = _predict(ag, obs, 0)
    for how, draw, ctr in (("draw", step, None), ("counter", M64, step - (1 << 31))):
        a1 = _predict(ag, obs, 1, draw=draw, ctr=ctr)
        torch.cuda.synchronize()
        assert torch.isfinite(a1).all(), f"{name} ({how}): {a1[row].tolist()}"
        if kind == "sac":
            assert (a1 >= ag.min_ac).all() and (a1 <= ag.max_ac).all()
            continue
        scale = (ag.max_ac - ag.min_ac) / 2 * float(ag.hps.actor_noise_std)
        zr = ((a1.double() - a0.double()) / scale.double()).cpu()
        # recovering z from two fp32 actions adds their rounding: 2 ulp(|a|) / (scale std)
        slack = (2 * 2.0 ** -23 * a1.abs().double().clamp_min(1.0) / scale.double()).cpu().numpy()
        zt, u1 = twin(key, step, stream, n, A, agent)
        tol = noise_tol(u1, zt) + slack
        dev = np.abs(zr.numpy() - zt)
        print(f"edge predict {name} ({how}): recovered z {zr[row, 2 * h:2 * h + 2].tolist()}, twin "
              f"{zt[row, 2 * h:2 * h + 2].tolist()}, worst dev/bound {float((dev / tol).max()):.3f}")
        assert (dev <= tol).all()


# ---------------------------------------------------------------------------------------------------- 4. behaviour policy
def _predict(owner, obs, mode, eps=None, draw=1, ctr=None):
    """b2rl_actor_predict for an Agent or a Population (obs [n, O] or [N, n, O]); ctr: counters[:, CTR_Q] for draw = ~0."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    stacked = hasattr(owner, "N")
    if stacked:
        args = L.UpdateArgs.from_buffer_copy(owner.args)
    else:
        args = L.UpdateArgs()
        args.hp, args.fmt, args.actor = owner._hyper, owner.fmt, owner.layout.actor.c_struct()
        args.arena, args.region_stride = owner.arena.flat.data_ptr(), owner.layout.region
        args.agent_base = owner.agent_id
        args.min_ac, args.max_ac = owner.min_ac.data_ptr(), owner.max_ac.data_ptr()
        args.counters = owner.counters.data_ptr()
    if ctr is not None:
        owner.counters[..., L.CTR_Q] = torch.as_tensor(ctr, dtype=torch.int64)
    n = obs.shape[-2]
    act = torch.empty(*obs.shape[:-1], owner.ac_dim, dtype=torch.float32, device="cuda")
    args.eps = L.ptr(eps)
    std = float(owner.hps.actor_noise_std) if owner.td3 else 0.0
    L.check(owner._lib.b2rl_actor_predict(C.byref(args), obs.data_ptr(), n, mode, std, C.c_uint64(draw), act.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream), "actor_predict")
    return act


def policy_ref(p, obs, A, td3, ln, lo, hi, std, z=None):
    """float64 behaviour policy (agents/nets.py): TD3 tanh(u) scale + bias (+ z scale std, no clamp); SAC mode
    tanh(mu) scale + bias, sample tanh(mu + sigma z) scale + bias, sigma = exp(-5 + 3.5 (tanh(raw log-std) + 1)).
    Returns (actions, d action / d z)."""
    u = mlp_forward({k: v.double() for k, v in p.items()}, obs.double(), ln)
    lo, hi = lo.double(), hi.double()
    scale, bias = (hi - lo) / 2, (hi + lo) / 2
    if td3:
        a = torch.tanh(u) * scale + bias
        return (a, None) if z is None else (a + z * scale * std, (scale * std).expand_as(a))
    mu, raw = u[..., :A], u[..., A:2 * A]
    sigma = torch.exp(-5.0 + 3.5 * (torch.tanh(raw) + 1.0))
    if z is None:
        return torch.tanh(mu) * scale + bias, None
    return torch.tanh(mu + sigma * z) * scale + bias, scale * sigma


def check_policy(what, got, want, dadz=None, z=None, ztol=None, rtol=1e-5, atol=2e-6):
    """|got - want| <= atol + rtol (|want| + |d action / d z * z|) (+ ztol |d action / d z| for device noise: tanh' <= 1).
    The noise term sigma z (SAC) / scale std z (TD3) is an fp32 product whose factor sigma = exp(log-std) carries the
    forward pass's relative error (times 3.5 through the log-std squash): it gets the same rtol as the action itself."""
    got = got.double().cpu()
    want = want.cpu()
    bound = atol + rtol * want.abs()
    if z is not None:
        bound = bound + rtol * (dadz * z).abs().cpu()
    if ztol is not None:
        bound = bound + torch.as_tensor(ztol) * dadz.abs().cpu()
    dev = (got - want).abs()
    ratio = float((dev / bound).max())
    print(f"{what}: worst |da| {float(dev.max()):.2e}, worst dev/bound {ratio:.3f}")
    assert torch.isfinite(got).all() and ratio <= 1.0, what


def _perturbed_actor(ag, gen):
    """The arena's actor with non-trivial biases and LayerNorm affine parameters (the reference init has zeros / ones)."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    lay = ag.layout
    named = lambda net: {k: v.detach().clone().cpu() for k, v in ag.arena.named(net, L.REGION_P).items()}
    actor = named(lay.actor)
    for k, v in actor.items():
        if k.endswith("bias"):
            v += 0.1 * torch.randn(v.shape, generator=gen)
        elif ".ln.weight" in k:
            v += 0.2 * torch.randn(v.shape, generator=gen)
    ag.load_params(actor, named(lay.critic[0]), named(lay.critic[1]))
    return {k: v.to("cuda") for k, v in actor.items()}


N_ROWS = (1, 7, 8, 9, 257, 5000)


@pytest.mark.gpu
@pytest.mark.parametrize("ln", [True, False], ids=["ln", "noln"])
@pytest.mark.parametrize("kind", ["sac", "td3"])
@pytest.mark.parametrize("ob", [1, 11, 32, 33, 376])
def test_behaviour_policy_matches_float64(ob, kind, ln):
    """b2rl_actor_predict against a float64 forward pass on the arena's (perturbed) parameters, with asymmetric
    per-dimension bounds: mode 0; mode 1 with host eps; mode 1 with device noise as a host-counted draw (key ~seed) and as
    draw = ~0 keyed on counters[CTR_Q] | 2^31. ob = 32 / 33 straddles W1S_ROWS (staged / streamed first layer); n covers
    ragged 8-row tiles and many row blocks. Device-noise bound: the host bound + the noise bound times scale * std (TD3)
    or scale * sigma (SAC)."""
    seed = SEED_HI ^ ob
    for A in (1, 3, 4, 5, 17):
        gen = torch.Generator().manual_seed(1000 * ob + A)
        lo = -0.5 - torch.rand(A, generator=gen)
        hi = 0.2 + 1.5 * torch.rand(A, generator=gen)
        ag = _agent(kind, A, ob=ob, seed=seed, layer_norm=ln, lo=lo.tolist(), hi=hi.tolist(), cache=False)
        ag.agent_id = 3 + A
        p = _perturbed_actor(ag, gen)
        obs = torch.randn(max(N_ROWS), ob, generator=gen).cuda()
        eps = torch.randn(max(N_ROWS), A, generator=gen).cuda()
        lo_d, hi_d = ag.min_ac.double(), ag.max_ac.double()
        std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
        want0, _ = policy_ref(p, obs, A, ag.td3, ln, lo_d, hi_d, std)
        want_h, dadz_h = policy_ref(p, obs, A, ag.td3, ln, lo_d, hi_d, std, eps.double())
        draw, ctr = 0x1234 + A, (1 << 31) + (1 << 32) * A + 77  # (bit 31 already set: | 2^31 leaves it)
        dev_noise = {}
        for how, step in (("draw", draw), ("counter", (ctr | (1 << 31)) & 0xFFFFFFFF)):
            z, u1 = twin(seed ^ M64, step, STREAM_ACTOR_EPS, max(N_ROWS), A, ag.agent_id)
            zt = torch.as_tensor(z, dtype=torch.float64, device="cuda")
            dev_noise[how] = policy_ref(p, obs, A, ag.td3, ln, lo_d, hi_d, std, zt), zt, noise_tol(u1, z)
        for n in N_ROWS:
            tag = f"predict {kind} ob={ob} A={A} ln={int(ln)} n={n}"
            check_policy(tag + " mode 0", _predict(ag, obs[:n], 0), want0[:n])
            check_policy(tag + " mode 1 host eps", _predict(ag, obs[:n], 1, eps=eps[:n]), want_h[:n], dadz_h[:n], eps[:n].double())
            for how in ("draw", "counter"):
                (want, dadz), zt, ztol = dev_noise[how]
                got = _predict(ag, obs[:n], 1, draw=draw) if how == "draw" else _predict(ag, obs[:n], 1, draw=M64, ctr=ctr)
                check_policy(f"{tag} mode 1 device noise ({how})", got, want[:n], dadz[:n], zt[:n], ztol[:n])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["sac", "td3"])
def test_stacked_behaviour_policy_matches_float64(kind):
    """N = 3 agents in grid y with agent_base = 5: agent g reads its own actor, observations and counters[g][CTR_Q] and
    keys its noise on global id 5 + g."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ids, A, ob, n, seed = [5, 6, 7], 6, 11, 37, 0xFFFFFFFF00000001
    lo, hi = [-1.0, -0.5, -2.0, -0.25, -1.0, -3.0], [1.0, 1.5, 0.5, 0.25, 2.0, 0.0]
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, ob, A, lo, hi, _hps(kind), "cuda", seed=seed, rb_capacity=64, use_graphs=False)
    gen = torch.Generator().manual_seed(42)
    obs = torch.randn(3, n, ob, generator=gen).cuda()
    eps = torch.randn(3, n, A, generator=gen).cuda()
    ctr = [(1 << 31) + 4, 9, (1 << 40) + 1]
    std = float(pop.hps.actor_noise_std) if pop.td3 else 0.0
    got = {"mode 0": _predict(pop, obs, 0), "host eps": _predict(pop, obs, 1, eps=eps),
           "draw": _predict(pop, obs, 1, draw=77), "counter": _predict(pop, obs, 1, draw=M64, ctr=ctr)}
    torch.cuda.synchronize()
    lo_d, hi_d = pop.min_ac.double(), pop.max_ac.double()
    for g in range(3):
        p = {k: v.clone() for k, v in pop.arena.named(pop.layout.actor, L.REGION_P, g).items()}
        want0, _ = policy_ref(p, obs[g], A, pop.td3, True, lo_d, hi_d, std)
        check_policy(f"stacked {kind} g={g} mode 0", got["mode 0"][g], want0)
        want, dadz = policy_ref(p, obs[g], A, pop.td3, True, lo_d, hi_d, std, eps[g].double())
        check_policy(f"stacked {kind} g={g} host eps", got["host eps"][g], want, dadz, eps[g].double())
        for how, step in (("draw", 77), ("counter", (ctr[g] | (1 << 31)) & 0xFFFFFFFF)):
            z, u1 = twin(seed ^ M64, step, STREAM_ACTOR_EPS, n, A, ids[g])
            zt = torch.as_tensor(z, dtype=torch.float64, device="cuda")
            want, dadz = policy_ref(p, obs[g], A, pop.td3, True, lo_d, hi_d, std, zt)
            check_policy(f"stacked {kind} g={g} device noise ({how})", got[how][g], want, dadz, zt, noise_tol(u1, z))
        assert int(pop.counters[g, L.CTR_Q]) == ctr[g]  # (the policy reads the counter, it does not advance it)


@pytest.mark.gpu
def test_behaviour_policy_fixture_cases_match_float64():
    """The golden cases' actors (reference initialisation, symmetric bounds, layer norm) on 7 stored observations with
    the cases' critic noise: mode 0 and mode 1 against float64, for sac_hopper, td3_hopper and sac_humanoid."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from tests.golden.cases import case_inputs
    from tests.helpers import make_agent
    for name in ("sac_hopper", "td3_hopper", "sac_humanoid"):
        inp = case_inputs(name)
        ag = make_agent(inp)
        obs = inp["storage"]["observations"][:7].float().cuda()
        eps = inp["eps_q"][0][:7].float().cuda()
        p = {k: v.clone() for k, v in ag.arena.named(ag.layout.actor, L.REGION_P).items()}
        std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
        ln, lo, hi = bool(ag.hps.layer_norm), ag.min_ac.double(), ag.max_ac.double()
        check_policy(f"{name} mode 0", ag.predict_device(obs, explore=False),
                     policy_ref(p, obs, ag.ac_dim, ag.td3, ln, lo, hi, std)[0])
        want, dadz = policy_ref(p, obs, ag.ac_dim, ag.td3, ln, lo, hi, std, eps.double())
        check_policy(f"{name} mode 1", ag.predict_device(obs, explore=True, eps=eps), want, dadz, eps.double())
