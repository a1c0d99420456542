"""Per-agent hyperparameters of a Population (include/b2rl.h b2rl_agent_hp_t): a swept population equals separate
populations built with each agent's values as plain hps, bitwise; every table field reaches its own agent and no other;
set_agent_hps and exploit (population-based training) change state without recapturing a graph; bad sweeps are refused.
Hopper shapes (O = 11, A = 3), batch 32, four agents."""
import ctypes as C
import math
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions

REPO = Path(__file__).resolve().parent.parent
OB, AC, B, CAP = 11, 3, 32, 1000

# every key differs between every pair of agents; agent 0 does not clip (clip_norm = 0), the others clip hard enough for
# the clip factor to be < 1 in the first actor steps; agent 1 has no target smoothing noise (td3_std = 0)
SWEEP = {
    "qnets_lr": [1e-3, 5e-4, 2e-3, 3e-4],
    "actor_lr": [3e-4, 1e-3, 1e-4, 6e-4],
    "log_alpha_lr": [1e-3, 3e-3, 5e-4, 2e-3],
    "gamma": [0.99, 0.95, 0.9, 0.999],
    "polyak": [0.005, 0.05, 0.1, 0.02],
    "td3_std": [0.2, 0.0, 0.4, 0.1],
    "td3_c": [0.5, 0.3, 0.1, 0.25],
    "clip_norm": [0.0, 0.05, 0.01, 0.002],
    "actor_noise_std": [0.1, 0.3, 0.05, 0.2],
    "alpha_init": [0.2, 0.5, 0.05, 1.0],
    "targ_ent": [-3.0, -1.0, 0.5, -6.0],
}
WIDE_SWEEP = dict(SWEEP, clip_norm=[0.0] * 4)
# a second value for agent 2, per key, with a visible effect within the run
PERTURB = {"qnets_lr": 4e-3, "actor_lr": 2e-3, "log_alpha_lr": 1e-2, "gamma": 0.5, "polyak": 0.3, "td3_std": 0.05,
           "td3_c": 0.02, "clip_norm": 1e-4, "actor_noise_std": 0.5, "alpha_init": 2.0, "targ_ent": -0.5}
# the keys a SAC / TD3 learner reads (the others are stored but have no effect on that algorithm)
USED = {"sac": ["qnets_lr", "actor_lr", "log_alpha_lr", "gamma", "polyak", "clip_norm", "alpha_init", "targ_ent"],
        "td3": ["qnets_lr", "actor_lr", "gamma", "polyak", "td3_std", "td3_c", "clip_norm", "actor_noise_std"]}


def _hps(algo, **over):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    return (sac_hps if algo == "sac" else td3_hps)(batch_size=B, **over)


def _data(agent_id, n=600):
    return make_synthetic_transitions(n, OB, AC, [-1.0] * AC, [1.0] * AC, seed=77 + agent_id)


def _pop(ids, algo, agent_hps=None, use_graphs=True, wide=None, **over):
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, OB, AC, [-1.0] * AC, [1.0] * AC, _hps(algo, **over), "cuda", seed=42, rb_capacity=CAP,
                     use_graphs=use_graphs, wide=wide, agent_hps=agent_hps)
    for g, aid in enumerate(ids):
        pop.fill_replay(_data(aid), agent=g)
    return pop


def _column(sweep, g):
    return {k: v[g] for k, v in sweep.items()}


def _separate(g, algo, sweep, **kw):
    """One-agent population with global id g and agent g's values as its plain hps."""
    return _pop([g], algo, **kw, **_column(sweep, g))


def _assert_agent_equal(pop, g, one, j=0):
    assert torch.equal(pop.arena.flat[g], one.arena.flat[j]), f"agent {g}: arena differs"
    sl = [0, 2, 3] if pop.wide else slice(None)  # (log alpha and its Adam moments, as test_gpu_population compares the wide path)
    assert torch.equal(pop.alpha_state[g, sl], one.alpha_state[j, sl]), f"agent {g}: alpha_state differs"
    assert torch.equal(pop.counters[g], one.counters[j]), f"agent {g}: counters differ"
    assert torch.equal(pop.out[g], one.out[j]), f"agent {g}: log block differs"


def _inputs(n_agents, n_it, n_new=4, n_obs=4, seed=3):
    from sac_td3_cudagraphs_pytorch_b200.replay import row_format
    rs = row_format(OB, AC).row_stride
    gen = torch.Generator().manual_seed(seed)
    return [(torch.randn(n_agents, n_new, rs, generator=gen), torch.randn(n_agents, n_obs, OB, generator=gen))
            for _ in range(n_it)]


def _run_steps(pop, inputs, pipelined=False, before=None):
    """step_async over the inputs; before(i) runs before step i is launched. Returns the actions of every step."""
    acts, prev = [], None
    for i, (rows, obs) in enumerate(inputs):
        if before is not None:
            before(i)
        pop.host_rows(rows.shape[1]).copy_(rows)
        pop.host_obs(obs.shape[1]).copy_(obs)
        t = pop.step_async(i, rows.shape[1], n_obs=obs.shape[1])
        acts.append(pop.wait_actions().copy())
        if pipelined:
            if prev is not None:
                pop.wait(prev)
            prev = t
        else:
            pop.wait(t)
    if pipelined and prev is not None:
        pop.wait(prev)
    torch.cuda.synchronize()
    return np.stack(acts)


# ---- 1. sweep == separate configurations, bitwise (row path) --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
@pytest.mark.parametrize("use_graphs", [True, False])
def test_sweep_equals_separate_configurations(algo, use_graphs):
    ids, n_it = [0, 1, 2, 3], 7
    pop = _pop(ids, algo, SWEEP, use_graphs=use_graphs)
    for _ in range(n_it):
        pop.iteration()
    torch.cuda.synchronize()
    assert torch.isfinite(pop.out).all()
    for g in ids:
        one = _separate(g, algo, SWEEP, use_graphs=use_graphs)
        for _ in range(n_it):
            one.iteration()
        torch.cuda.synchronize()
        _assert_agent_equal(pop, g, one)
        assert pop.agent_hps(g) == pytest.approx(_column(SWEEP, g))
    if algo == "sac":  # alpha_init reached the device
        assert len(set(pop.alpha_state[:, 0].tolist())) == 4


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
@pytest.mark.parametrize("pipelined", [False, True])
def test_swept_steps_equal_separate_configurations(algo, pipelined):
    """The step graph: behaviour policy (explore_std), replay write and iteration."""
    ids, inputs = [0, 1, 2, 3], _inputs(4, 7)
    pop = _pop(ids, algo, SWEEP)
    acts = _run_steps(pop, inputs, pipelined)
    for g in ids:
        one = _separate(g, algo, SWEEP)
        a1 = _run_steps(one, [(r[g:g + 1], o[g:g + 1]) for r, o in inputs], pipelined)
        _assert_agent_equal(pop, g, one)
        assert torch.equal(pop.storage[g], one.storage[0])
        assert np.array_equal(acts[:, g], a1[:, 0]), f"agent {g}: actions differ"


# ---- 2. the 3xTF32 tensor-core path --------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_wide_sweep_equals_separate_configurations(algo):
    ids, n_it = [0, 1, 2, 3], 7
    pop = _pop(ids, algo, WIDE_SWEEP, wide="3xtf32")
    for _ in range(n_it):
        pop.iteration()
    torch.cuda.synchronize()
    assert torch.isfinite(pop.out).all()
    for g in ids:
        one = _separate(g, algo, WIDE_SWEEP, wide="3xtf32")
        for _ in range(n_it):
            one.iteration()
        torch.cuda.synchronize()
        _assert_agent_equal(pop, g, one)


@pytest.mark.gpu
@pytest.mark.parametrize("wide", [None, "3xtf32"])
def test_swept_population_is_invariant_to_sharding(wide):
    sweep = WIDE_SWEEP if wide else SWEEP
    col = lambda ids: {k: [v[i] for i in ids] for k, v in sweep.items()}
    whole = _pop([0, 1, 2, 3], "sac", sweep, wide=wide)
    parts = [_pop([0, 1], "sac", col([0, 1]), wide=wide), _pop([2], "sac", col([2]), wide=wide, use_graphs=False),
             _pop([3], "sac", col([3]), wide=wide)]
    for _ in range(7):
        whole.iteration()
        for p in parts:
            p.iteration()
    torch.cuda.synchronize()
    assert torch.equal(whole.arena.flat, torch.cat([p.arena.flat for p in parts]))
    assert torch.equal(whole.counters, torch.cat([p.counters for p in parts]))
    assert torch.equal(whole.alpha_state, torch.cat([p.alpha_state for p in parts]))
    assert torch.equal(whole.out, torch.cat([p.out for p in parts]))


# ---- 3. every field reaches its agent and only its agent --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_every_field_reaches_its_agent_only(algo):
    inputs = _inputs(4, 7)
    ref = _pop([0, 1, 2, 3], algo, SWEEP)
    ref_acts = _run_steps(ref, inputs)
    for key in USED[algo]:
        sweep = {k: list(v) for k, v in SWEEP.items()}
        sweep[key][2] = PERTURB[key]
        pop = _pop([0, 1, 2, 3], algo, sweep)
        acts = _run_steps(pop, inputs)
        for g in (0, 1, 3):
            assert torch.equal(pop.arena.flat[g], ref.arena.flat[g]), f"{key}: agent {g} changed"
            assert torch.equal(pop.alpha_state[g], ref.alpha_state[g]), f"{key}: agent {g} changed"
            assert np.array_equal(acts[:, g], ref_acts[:, g]), f"{key}: agent {g}'s actions changed"
        changed = (not torch.equal(pop.arena.flat[2], ref.arena.flat[2]) or not torch.equal(pop.alpha_state[2], ref.alpha_state[2])
                   or not np.array_equal(acts[:, 2], ref_acts[:, 2]))  # (explore_std shows in the actions only)
        assert changed, f"{key}: agent 2's value had no effect"


# ---- 4. mixed clipping ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_unclipped_member_of_a_clipping_population_equals_an_unclipped_learner(algo):
    pop = _pop([0, 1, 2, 3], algo, SWEEP)
    assert pop._clip and pop.agent_hps(0)["clip_norm"] == 0.0
    assert math.isinf(float(pop.agent_hp_table[0, 8]))  # the +inf encoding
    one = _separate(0, algo, SWEEP)
    assert not one._clip  # the separate learner runs the unclipped step (no sumsq launch, seg.clip = 0)
    for _ in range(7):
        pop.iteration()
        one.iteration()
    torch.cuda.synchronize()
    _assert_agent_equal(pop, 0, one)
    # and clipping did happen for the others: an unclipped twin of agent 3 ends elsewhere
    free = _pop([3], algo, None, **dict(_column(SWEEP, 3), clip_norm=0.0))
    for _ in range(7):
        free.iteration()
    torch.cuda.synchronize()
    assert not torch.equal(pop.arena.flat[3], free.arena.flat[0])


# ---- 5. set_agent_hps mid-run ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
@pytest.mark.parametrize("pipelined", [False, True])
def test_set_agent_hps_mid_run_equals_separate_learners_given_the_same_change(algo, pipelined):
    change = {"gamma": 0.8, "actor_lr": 2e-3, "polyak": 0.2, "clip_norm": 0.0, "actor_noise_std": 0.4, "targ_ent": -2.0}
    inputs = _inputs(4, 8)
    pop = _pop([0, 1, 2, 3], algo, SWEEP)
    n_graphs = []

    def before(i):
        if i == 4:
            n_graphs.append(len(pop.graphs))
            pop.set_agent_hps([1, 2], **change)
            n_graphs.append(len(pop.graphs))
    acts = _run_steps(pop, inputs, pipelined, before)
    assert n_graphs[0] == n_graphs[1] and n_graphs[0] > 0
    assert pop.agent_hps(2)["gamma"] == pytest.approx(0.8) and pop.agent_hps(0)["gamma"] == pytest.approx(0.99)
    for g in (0, 2):
        one = _separate(g, algo, SWEEP)
        a1 = _run_steps(one, [(r[g:g + 1], o[g:g + 1]) for r, o in inputs], pipelined,
                        (lambda i: one.set_agent_hps(0, **change) if i == 4 else None) if g == 2 else None)
        _assert_agent_equal(pop, g, one)
        assert np.array_equal(acts[:, g], a1[:, 0])


# ---- 6. exploit ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
@pytest.mark.parametrize("wide", [None, "3xtf32"])
def test_exploit_copies_the_learner_state_and_keeps_the_replay(algo, wide):
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    sweep = WIDE_SWEEP if wide else SWEEP
    pop = _pop([0, 1, 2, 3], algo, sweep, wide=wide)
    pop.lo_mirror()  # (a 3xTF32 mirror, kept by the optimizer launches: exploit copies its row too)
    for _ in range(4):
        pop.iteration()
    torch.cuda.synchronize()
    before = {k: getattr(pop, k).clone() for k in ("storage", "counters", "alpha_state")}
    arena_before = pop.arena.flat.clone()
    lo = pop._lo.clone()
    pop.exploit(2, 0)
    torch.cuda.synchronize()
    assert torch.equal(pop.arena.flat[2], pop.arena.flat[0])
    assert torch.equal(pop.alpha_state[2], pop.alpha_state[0])
    assert torch.equal(pop.counters[2, :3], pop.counters[0, :3])
    assert torch.equal(pop.agent_hp_table[2], pop.agent_hp_table[0])
    assert pop.agent_hps(2) == pop.agent_hps(0)
    assert torch.equal(pop._lo[2], pop._lo[0])
    assert torch.equal(pop.storage, before["storage"])
    assert torch.equal(pop.counters[2, 3:], before["counters"][2, 3:])  # SAMPLE, tickets, SIZE, CURSOR stay agent 2's
    for g in (0, 1, 3):
        assert torch.equal(pop.arena.flat[g], arena_before[g])
        assert torch.equal(pop.counters[g], before["counters"][g])
        assert torch.equal(pop.alpha_state[g], before["alpha_state"][g])
        assert torch.equal(pop._lo[g], lo[g])
    # k more steps == a one-agent population with global id 2 (its replay, its random streams) loaded with agent 0's state
    snap = (pop.arena.flat[0].clone(), pop.alpha_state[0].clone(), pop.counters[0, :3].clone())
    pop.set_agent_hps(2, gamma=0.97)
    for i in range(4, 9):  # (the same iteration indices: the actor-step cadence follows them)
        pop.iteration(i)
    one = _pop([2], algo, None, wide=wide, **dict(_column(sweep, 0), gamma=0.97))
    one.arena.flat[0].copy_(snap[0])
    one.alpha_state[0].copy_(snap[1])
    one.counters[0, :3].copy_(snap[2])
    one.lo_mirror()
    for i in range(4, 9):
        one.iteration(i)
    torch.cuda.synchronize()
    _assert_agent_equal(pop, 2, one)
    assert int(pop.counters[2, L.CTR_SIZE]) == int(before["counters"][2, L.CTR_SIZE])


# ---- 7. rejections ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_sweeps_and_calls_are_refused():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    with pytest.raises(L.B2rlError, match="batch_size"):
        _pop([0, 1], "sac", {"batch_size": [32, 64]})
    with pytest.raises(L.B2rlError, match="2 values"):
        _pop([0, 1], "sac", {"gamma": [0.9, 0.9, 0.9]})
    with pytest.raises(L.B2rlError, match="gamma"):
        _pop([0, 1], "sac", {"gamma": [0.9, 1.5]})
    with pytest.raises(L.B2rlError, match="clip_norm"):
        _pop([0, 1], "sac", {"clip_norm": [0.0, 1.0]}, wide="3xtf32")
    pop = _pop([0, 1, 2, 3], "sac", SWEEP)
    with pytest.raises(L.B2rlError, match="alpha_init"):
        pop.set_agent_hps(1, alpha_init=0.3)
    with pytest.raises(L.B2rlError, match="polyak"):
        pop.set_agent_hps(1, polyak=-0.1)
    with pytest.raises(L.B2rlError, match="local agent"):
        pop.set_agent_hps(4, gamma=0.9)
    with pytest.raises(L.B2rlError, match="same agent"):
        pop.exploit(1, 1)
    plain = _pop([0, 1], "sac", None)
    with pytest.raises(L.B2rlError, match="clip"):
        plain.set_agent_hps(0, clip_norm=1.0)  # its graphs have no clipped step
    # the fused-optimizer entry points refuse a table, before any launch (the arena stays as it is)
    lib, lay = L.load(), pop.layout
    opt = L.AdamArgs()
    opt.seg[0] = L.Seg(lay.critic[0].begin, lay.critic[1].end, 1e-3, 1, 0, L.CTR_Q, 1.0, 0)
    opt.n_seg, opt.n_agents, opt.beta1, opt.beta2, opt.eps = 1, 4, 0.9, 0.999, 1e-8
    opt.region_stride, opt.arena_agent_stride = lay.region, pop.arena.agent_stride
    opt.arena, opt.counters = pop.arena.flat.data_ptr(), pop.counters.data_ptr()
    snap = pop.arena.flat.clone()
    assert lib.b2rl_critic_update_opt(C.byref(pop._hp_args), C.byref(opt), None) == -1
    assert b"per-agent" in lib.b2rl_last_error()
    plain_args = pop.args  # (the population's own launches pass _hp_args, which carries the table)
    assert plain_args.agent_hp is None
    opt.agent_hp = pop.agent_hp_table.data_ptr()
    opt.seg[0] = L.Seg(lay.actor.begin, lay.actor.end, 1e-3, 1, 0, L.CTR_PI, 1.0, 0)
    assert lib.b2rl_actor_update_opt(C.byref(plain_args), C.byref(opt), None) == -1
    assert b"per-agent" in lib.b2rl_last_error()
    torch.cuda.synchronize()
    assert torch.equal(pop.arena.flat, snap)


# ---- 8. CPU: the ABI and the host function that builds the table -----------------------------------------------------------------
def test_agent_hp_struct_matches_the_c_compiler():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    fields = ["lr", "gamma", "polyak", "td3_std", "td3_c", "targ_ent", "clip_norm", "explore_std", "reserved"]
    exprs = ["sizeof(b2rl_agent_hp_t)"] + [f"__builtin_offsetof(b2rl_agent_hp_t, {f})" for f in fields] + [
        "__builtin_offsetof(b2rl_update_args_t, agent_hp)", "__builtin_offsetof(b2rl_adam_args_t, agent_hp)",
        "__builtin_offsetof(b2rl_stack_t, agent_hp)"]
    src = '#include <stdio.h>\n#include "b2rl.h"\nint main(){' + "".join(f'printf("%zu\\n", (size_t)({e}));' for e in exprs) + \
          "return 0;}"
    with tempfile.TemporaryDirectory() as d:
        c = Path(d) / "s.c"
        c.write_text(src)
        subprocess.check_call(["gcc", "-I", str(REPO / "include"), str(c), "-o", str(Path(d) / "s")])
        out = [int(x) for x in subprocess.check_output([str(Path(d) / "s")]).split()]
    want = [C.sizeof(L.AgentHp)] + [getattr(L.AgentHp, f).offset for f in fields] + [
        L.UpdateArgs.agent_hp.offset, L.AdamArgs.agent_hp.offset, L.Stack.agent_hp.offset]
    assert out == want
    assert out[0] == 64


def test_table_builder_values_and_encodings():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.population import agent_hp_table, agent_hp_values
    for algo in ("sac", "td3"):
        vals = agent_hp_values(_hps(algo), 4, AC, SWEEP)
        t = agent_hp_table(vals, algo == "td3")
        assert t.shape == (4, 16) and t.dtype == np.float32
        for g in range(4):
            r = L.AgentHp.from_buffer_copy(t[g].tobytes())
            assert r.lr[L.CTR_Q] == np.float32(SWEEP["qnets_lr"][g]) and r.lr[L.CTR_PI] == np.float32(SWEEP["actor_lr"][g])
            assert r.lr[L.CTR_ALPHA] == np.float32(SWEEP["log_alpha_lr"][g])
            assert (r.gamma, r.polyak, r.targ_ent) == tuple(np.float32(SWEEP[k][g]) for k in ("gamma", "polyak", "targ_ent"))
            cn = SWEEP["clip_norm"][g]
            assert r.clip_norm == (np.float32(cn) if cn > 0 else math.inf)
            if algo == "td3":
                assert (r.td3_std, r.td3_c, r.explore_std) == tuple(
                    np.float32(SWEEP[k][g]) for k in ("td3_std", "td3_c", "actor_noise_std"))
            else:  # SAC passes no TD3 noise, as the scalar path does
                assert (r.td3_std, r.td3_c, r.explore_std) == (0.0, 0.0, 0.0)
            assert list(r.reserved) == [0.0] * 6
    # defaults: hps, and targ_ent = -A; a sequence of override mappings is the same as the mapping form
    vals = agent_hp_values(_hps("sac"), 2, AC)
    assert vals[0] == vals[1] and vals[0]["targ_ent"] == -float(AC) and vals[0]["gamma"] == 0.99
    assert agent_hp_values(_hps("sac"), 2, AC, [{"gamma": 0.9}, {}]) == agent_hp_values(_hps("sac"), 2, AC, {"gamma": [0.9, 0.99]})
    assert agent_hp_values(_hps("sac", targ_ent=-1.5), 1, AC)[0]["targ_ent"] == -1.5


@pytest.mark.parametrize("sweep,wide,msg", [
    ({"batch_size": [32, 64]}, False, "'batch_size' cannot differ"),
    ({"actor_update_delay": [1, 2]}, False, "'actor_update_delay'"),
    ({"layer_norm": [True, False]}, False, "'layer_norm'"),
    ({"rb_capacity": [10, 20]}, False, "'rb_capacity'"),
    ([{"crit_targ_update_freq": 2}, {}], False, "'crit_targ_update_freq'"),
    ({"gamma": [0.9]}, False, "2 values"),
    ([{"gamma": 0.9}], False, "2 override mappings"),
    ({"gamma": [0.9, 0.0]}, False, r"gamma = 0.0 must be in \(0, 1\]"),
    ({"gamma": [0.9, 1.01]}, False, "gamma"),
    ({"polyak": [0.1, 1.5]}, False, r"polyak = 1.5 must be in \[0, 1\]"),
    ({"qnets_lr": [1e-3, -1e-3]}, False, "qnets_lr = -0.001 must be >= 0"),
    ({"td3_std": [0.1, -0.1]}, False, "td3_std"),
    ({"td3_c": [0.1, -0.1]}, False, "td3_c"),
    ({"clip_norm": [0.1, -1.0]}, False, "clip_norm"),
    ({"actor_noise_std": [0.1, -0.1]}, False, "actor_noise_std"),
    ({"alpha_init": [0.1, 0.0]}, False, "alpha_init"),
    ({"gamma": [0.9, float("nan")]}, False, "finite"),
    ({"clip_norm": [0.0, 1.0]}, True, "no gradient clipping"),
])
def test_table_builder_refuses_bad_sweeps(sweep, wide, msg):
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.population import agent_hp_values
    with pytest.raises(L.B2rlError, match=msg):
        agent_hp_values(_hps("sac"), 2, AC, sweep, wide=wide)
