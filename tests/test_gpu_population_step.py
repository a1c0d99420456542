"""The population trained against environments: the stacked behaviour policy (b2rl_actor_predict with n_agents > 1), the
stacked device-cursor replay write (b2rl_replay_extend_dev_stack) and Population.step_async — policy, replay write,
iteration and log block as one graph replay — equal, bitwise, N separate learners driven through
LearnerEngine.step_async, do not depend on sharding or on pipelining, and reject bad calls loudly."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions

IDS = [5, 6, 7]
UINT64_MAX = 2 ** 64 - 1


def _L():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    return L


def _hps(algo, B=32):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    return (sac_hps if algo == "sac" else td3_hps)(batch_size=B)


def _data(agent_id, n, ob=11, ac=3):
    return make_synthetic_transitions(n, ob, ac, [-1.0] * ac, [1.0] * ac, seed=77 + agent_id)


def _population(ids, algo, n0, cap, B=32, wide=None, use_graphs=True, ob=11, ac=3):
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, ob, ac, [-1.0] * ac, [1.0] * ac, _hps(algo, B), "cuda", seed=42, rb_capacity=cap,
                     use_graphs=use_graphs, wide=wide)
    if n0:
        for g, aid in enumerate(ids):
            pop.fill_replay(_data(aid, n0, ob, ac), agent=g)
    return pop


def _inputs(n_agents, n_it, n_new, n_obs, rs, ob=11, seed=3):
    """Per step: new transitions [N, n_new, row_stride] and observations [N, n_obs, ob] (host tensors)."""
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(n_agents, n_new, rs, generator=g), torch.randn(n_agents, n_obs, ob, generator=g)) for _ in range(n_it)]


def _run_steps(pop, inputs, pipelined=False):
    """Drive step_async with the given inputs; returns (log blocks, actions) per step. pipelined: one step in flight (the
    host fills the other staging slot and launches step t before it reads step t - 1's log block)."""
    logs, acts, prev = [], [], None
    for i, (rows, obs) in enumerate(inputs):
        n_new, n_obs = rows.shape[1], obs.shape[1]
        pop.host_rows(n_new).copy_(rows)
        pop.host_obs(n_obs).copy_(obs)
        t = pop.step_async(i, n_new, n_obs=n_obs)
        acts.append(pop.wait_actions().copy())
        if pipelined:
            if prev is not None:
                logs.append(pop.wait(prev).clone())
            prev = t
        else:
            logs.append(pop.wait(t).clone())
    if pipelined:
        logs.append(pop.wait(prev).clone())
    torch.cuda.synchronize()
    return logs, acts


def _same_state(a, b):
    assert torch.equal(a.arena.flat, b.arena.flat)
    assert torch.equal(a.counters, b.counters)
    assert torch.equal(a.alpha_state, b.alpha_state)
    assert torch.equal(a.storage, b.storage)
    assert (a.cursor, a.size) == (b.cursor, b.size)


# ---- 1. the stacked replay write ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ob,ac", [(11, 3), (376, 17)])  # Hopper rows: 7 16-byte chunks; Humanoid rows: 193
@pytest.mark.parametrize("pinned", [False, True])
def test_stacked_replay_write_equals_per_agent_writes(ob, ac, pinned):
    L = _L()
    from sac_td3_cudagraphs_pytorch_b200.replay import row_format
    lib, st = L.load(), torch.cuda.current_stream().cuda_stream
    L.init_device("cuda")
    fmt = row_format(ob, ac)
    rs, N, cap = fmt.row_stride, 3, 50
    assert rs // 4 == (7 if ob == 11 else 193)
    gen = torch.Generator().manual_seed(1)
    ref = torch.randn(N, cap, rs, generator=gen)
    stacked, single = ref.cuda(), ref.cuda()
    ctr = torch.zeros(N, 8, dtype=torch.int64)
    ctr[:, L.CTR_CURSOR] = torch.tensor([40, 45, 3])  # every agent has its own cursor and fill count
    ctr[:, L.CTR_SIZE] = torch.tensor([40, 50, 3])
    c_stacked, c_single, c_ref = ctr.cuda(), ctr.cuda(), ctr.clone()
    for n in (7, 20, 1, cap):  # 40 + 7 + 20 wraps; n = capacity rewrites every row
        rows = torch.randn(N, n, rs, generator=gen)
        src = rows.pin_memory() if pinned else rows.cuda()
        L.check(lib.b2rl_replay_extend_dev_stack(stacked.data_ptr(), stacked[0].numel(), cap, fmt, src.data_ptr(), n, N,
                                                 c_stacked.data_ptr(), st), "extend_dev_stack")
        for g in range(N):
            L.check(lib.b2rl_replay_extend_dev(single[g].data_ptr(), cap, fmt, src[g].data_ptr(), n, c_single[g].data_ptr(), st),
                    "extend_dev")
        for g in range(N):  # host model: torchrl's round-robin writer, per agent
            cur = int(c_ref[g, L.CTR_CURSOR])
            ref[g, (cur + torch.arange(n)) % cap] = rows[g]
            c_ref[g, L.CTR_CURSOR] = (cur + n) % cap
            c_ref[g, L.CTR_SIZE] = min(cap, int(c_ref[g, L.CTR_SIZE]) + n)
        torch.cuda.synchronize()
        assert torch.equal(stacked, single)
        assert torch.equal(c_stacked, c_single)
        assert torch.equal(stacked.cpu(), ref)
        assert torch.equal(c_stacked.cpu(), c_ref)
        assert (c_stacked[:, L.CTR_XTICKET] == 0).all()


# ---- 2. the stacked behaviour policy -----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
@pytest.mark.parametrize("ob,ac", [(11, 3), (376, 17)])  # both predict_kernel instantiations (staged / streamed first layer)
def test_stacked_policy_equals_per_agent_policy(algo, ob, ac):
    L = _L()
    pop = _population(IDS, algo, 0, 16, ob=ob, ac=ac)
    lib, st = pop._lib, torch.cuda.current_stream().cuda_stream
    pop.counters[:, L.CTR_Q] = torch.tensor([3, 9, 1])  # keys of the draw = UINT64_MAX noise, per agent
    std = float(pop.hps.actor_noise_std) if pop.td3 else 0.0
    gen = torch.Generator().manual_seed(2)
    for n in (5, 9):  # a ragged row block; two row blocks
        obs = torch.randn(len(IDS), n, ob, generator=gen).cuda()
        for mode in (0, 1):
            for draw in (7, UINT64_MAX):
                got = torch.full((len(IDS), n, ac), float("nan"), device="cuda")
                L.check(lib.b2rl_actor_predict(C.byref(pop.args), obs.data_ptr(), n, mode, std, C.c_uint64(draw),
                                               got.data_ptr(), st), "stacked predict")
                for g, aid in enumerate(IDS):
                    one = L.UpdateArgs.from_buffer_copy(pop.args)
                    one.n_agents, one.agent_base = g % 2, aid  # 0 (Agent.predict_device) and 1 both mean one learner
                    one.arena, one.counters = pop.arena.flat[g].data_ptr(), pop.counters[g].data_ptr()
                    want = torch.full((n, ac), float("nan"), device="cuda")
                    L.check(lib.b2rl_actor_predict(C.byref(one), obs[g].data_ptr(), n, mode, std, C.c_uint64(draw),
                                                   want.data_ptr(), st), "single predict")
                    torch.cuda.synchronize()
                    assert torch.equal(got[g], want), (n, mode, draw, aid)
                assert torch.isfinite(got).all()
                assert not torch.equal(got[0], got[1])  # own parameters (and noise) per agent


# ---- 3. the population step = N separate learners --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_population_step_equals_separate_learner_steps(algo):
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.population import init_agent_params
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    n0, cap, n_new, n_obs, n_it = 200, 230, 4, 5, 12  # 200 + 12 x 4 > 230: every agent's cursor wraps
    pop = _population(IDS, algo, n0, cap)
    inputs = _inputs(len(IDS), n_it, n_new, n_obs, pop.fmt.row_stride)
    logs, acts = _run_steps(pop, inputs)
    hps = _hps(algo)
    lo, hi = torch.full((3,), -1.0), torch.full((3,), 1.0)
    for g, aid in enumerate(IDS):
        rb = ReplayBuffer(cap, "cuda", seed=42, agent_id=aid)
        rb.extend({k: v.cuda() for k, v in _data(aid, n0).items()})
        ag = Agent({"ob_shape": (11,), "ac_shape": (3,)}, lo.numpy(), hi.numpy(), torch.device("cuda"), hps, rb=rb,
                   seed=42, agent_id=aid)
        ag.load_params(*init_agent_params(aid, 42, 11, 3, algo == "td3", True, lo, hi))
        eng = LearnerEngine(ag, use_graphs=True)
        for i, (rows, obs) in enumerate(inputs):
            eng.host_rows(n_new).copy_(rows[g])
            eng.host_obs(n_obs).copy_(obs[g])
            t = eng.step_async(i, n_new, n_obs=n_obs)
            a = eng.wait_actions().copy()
            out = eng.wait(t).clone()
            assert np.array_equal(acts[i][g], a), f"agent {aid}: actions differ at step {i}"
            assert torch.equal(logs[i][g], out), f"agent {aid}: log block differs at step {i}"
        torch.cuda.synchronize()
        assert torch.equal(pop.arena.flat[g], ag.arena.flat[0]), f"agent {aid}: stacked != separate"
        assert torch.equal(pop.counters[g], ag.counters)
        assert torch.equal(pop.alpha_state[g, :4], ag._alpha_state[:4])
        assert torch.equal(pop.storage[g], rb.storage)
    assert pop.cursor == rb._cursor == (n0 + n_it * n_new) % cap and pop.size == cap
    assert not torch.equal(pop.arena.flat[0], pop.arena.flat[1])
    assert all(np.isfinite(a).all() for a in acts) and all(torch.isfinite(o).all() for o in logs)


# ---- 4. pipelined = synchronous --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_pipelined_population_steps_equal_synchronous_steps(algo):
    n0, cap, n_new, n_obs, n_it = 200, 230, 4, 3, 13
    sync, pipe = _population(IDS, algo, n0, cap), _population(IDS, algo, n0, cap)
    inputs = _inputs(len(IDS), n_it, n_new, n_obs, sync.fmt.row_stride, seed=4)
    want_logs, want_acts = _run_steps(sync, inputs)
    got_logs, got_acts = _run_steps(pipe, inputs, pipelined=True)
    for i in range(n_it):
        assert torch.equal(got_logs[i], want_logs[i]), f"log block differs at step {i}"
        assert np.array_equal(got_acts[i], want_acts[i]), f"actions differ at step {i}"
    _same_state(sync, pipe)


# ---- 5. shard invariance of the step, on both paths --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo,B,wide", [("sac", 32, None), ("td3", 32, None), ("sac", 200, "3xtf32"), ("td3", 200, "3xtf32")])
def test_population_step_is_invariant_to_sharding(algo, B, wide):
    """[0,1,2,3] on one GPU == [0,1] + [2] + [3], bitwise, actions included; B = 200 is ragged against the wide path's
    128-row tiles."""
    n0, cap, n_new, n_obs, n_it = 300, 330, 4, 5, 9
    whole = _population([0, 1, 2, 3], algo, n0, cap, B=B, wide=wide)
    parts = [_population(ids, algo, n0, cap, B=B, wide=wide) for ids in ([0, 1], [2], [3])]
    inputs = _inputs(4, n_it, n_new, n_obs, whole.fmt.row_stride, seed=5)
    w_logs, w_acts = _run_steps(whole, inputs)
    lo = 0
    p_logs, p_acts = [], []
    for p in parts:
        lg, ac = _run_steps(p, [(r[lo:lo + p.N], o[lo:lo + p.N]) for r, o in inputs])
        p_logs.append(lg)
        p_acts.append(ac)
        lo += p.N
    for i in range(n_it):
        assert torch.equal(w_logs[i], torch.cat([lg[i] for lg in p_logs])), f"log blocks differ at step {i}"
        assert np.array_equal(w_acts[i], np.concatenate([ac[i] for ac in p_acts])), f"actions differ at step {i}"
    assert torch.equal(whole.arena.flat, torch.cat([p.arena.flat for p in parts]))
    assert torch.equal(whole.counters, torch.cat([p.counters for p in parts]))
    assert torch.equal(whole.storage, torch.cat([p.storage for p in parts]))
    assert torch.isfinite(whole.out).all()


# ---- 6. the wide step = the eager wide path ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_wide_population_step_equals_eager_extend_plus_iteration(algo):
    L = _L()
    n0, cap, n_new, n_obs, n_it, B = 300, 330, 4, 5, 9, 200
    step = _population(IDS, algo, n0, cap, B=B, wide="3xtf32")
    eager = _population(IDS, algo, n0, cap, B=B, wide="3xtf32", use_graphs=False)
    inputs = _inputs(len(IDS), n_it, n_new, n_obs, step.fmt.row_stride, seed=6)
    logs, acts = _run_steps(step, inputs)
    std = float(eager.hps.actor_noise_std) if eager.td3 else 0.0
    st = torch.cuda.current_stream().cuda_stream
    for i, (rows, obs) in enumerate(inputs):
        obs_d = obs.cuda()
        a = torch.empty(len(IDS), n_obs, 3, device="cuda")  # the policy as the step runs it: noise keyed on the counters
        L.check(eager._lib.b2rl_actor_predict(C.byref(eager.args), obs_d.data_ptr(), n_obs, 1, std, C.c_uint64(UINT64_MAX),
                                              a.data_ptr(), st), "predict")
        eager.extend(rows.cuda())
        eager.iteration(i)
        torch.cuda.synchronize()
        assert np.array_equal(acts[i], a.cpu().numpy()), f"actions differ at step {i}"
        assert torch.equal(logs[i], eager.out.cpu()), f"log block differs at step {i}"
    _same_state(step, eager)


# ---- 7. collection before learning -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_collection_with_predict_and_extend_then_training(algo):
    """The reference loop from an empty buffer: predict + extend up to learning_starts (orchestrator.py:329-333), then the
    step graph trains every agent."""
    L = _L()
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    ids, n_env, learning_starts, cap = [0, 1, 2], 4, 64, 200
    pop = _population(ids, algo, 0, cap)
    N, gen = len(ids), torch.Generator().manual_seed(8)
    obs = torch.randn(N, n_env, 11, generator=gen)
    evals = [pop.predict(obs, explore=False) for _ in range(2)]
    assert torch.equal(evals[0], evals[1])  # evaluation episodes: deterministic
    while pop.size < learning_starts:
        act = pop.predict(obs, explore=True)
        again = pop.predict(obs, explore=True)
        assert not torch.equal(act, again)  # every call draws new exploration noise
        nxt = torch.randn(N, n_env, 11, generator=gen)
        td = {"observations": obs.reshape(-1, 11), "actions": act.cpu().reshape(-1, 3),
              "rewards": torch.randn(N * n_env, 1, generator=gen), "dones": torch.zeros(N * n_env, 1, dtype=torch.bool),
              "next_observations": nxt.reshape(-1, 11)}
        pop.extend(pack_rows(td, pop.fmt).reshape(N, n_env, -1).pin_memory())
        torch.cuda.synchronize()  # (the pinned source of an eager extend must outlive the write)
        obs = nxt
    assert pop.size == learning_starts and pop.cursor == learning_starts
    assert (pop.counters[:, L.CTR_SIZE] == learning_starts).all() and (pop.counters[:, L.CTR_CURSOR] == learning_starts).all()
    before = pop.arena.flat[:, L.REGION_P].clone()
    for i in range(10):
        pop.host_rows(n_env).normal_(generator=gen)
        pop.host_obs(n_env).copy_(torch.randn(N, n_env, 11, generator=gen))
        out = pop.step(i, n_env, n_obs=n_env)
        assert out.shape == (N, 8) and torch.isfinite(out[:, :2]).all()
        assert np.isfinite(pop.wait_actions()).all()
    torch.cuda.synchronize()
    assert pop.size == learning_starts + 10 * n_env == int(pop.counters[0, L.CTR_SIZE])
    assert all(not torch.equal(before[g], pop.arena.flat[g, L.REGION_P]) for g in range(N))


# ---- 8. errors are loud ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_population_step_rejects_bad_calls():
    L = _L()
    pop = _population(IDS, "sac", 50, 60)
    with pytest.raises(L.B2rlError):
        pop.step_async(0, n_new=61)  # more transitions than the replay holds
    with pytest.raises(L.B2rlError):
        pop.extend(torch.zeros(len(IDS) - 1, 4, pop.fmt.row_stride, device="cuda"))  # wrong number of agents
    with pytest.raises(L.B2rlError):
        pop.extend(torch.zeros(len(IDS), 4, pop.fmt.row_stride - 4, device="cuda"))  # wrong row width
    with pytest.raises(L.B2rlError):
        pop.extend(torch.zeros(len(IDS), 61, pop.fmt.row_stride, device="cuda"))  # n > capacity
    with pytest.raises(L.B2rlError):
        pop.predict(torch.zeros(len(IDS), 4, 12), explore=True)  # wrong observation width
    with pytest.raises(L.B2rlError):
        pop.predict(torch.zeros(4, 11), explore=True)  # no agent dimension
    with pytest.raises(L.B2rlError):
        pop.predict(torch.zeros(len(IDS), 4, 11), explore=True, eps=torch.zeros(len(IDS), 4, 2))
    eager = _population(IDS, "sac", 50, 60, use_graphs=False)
    with pytest.raises(L.B2rlError):
        eager.step_async(0, 4)
    with pytest.raises(L.B2rlError):
        eager.wait_actions()  # no step has published actions
    torch.cuda.synchronize()
    assert (pop.counters[:, L.CTR_SIZE] == 50).all() and pop.size == 50  # nothing was written


def test_stacked_entry_points_reject_bad_arguments_before_any_launch():
    """Argument checks of the C ABI (no GPU needed: the calls fail before anything is enqueued)."""
    L = _L()
    from sac_td3_cudagraphs_pytorch_b200.arena import make_layout
    from sac_td3_cudagraphs_pytorch_b200.replay import row_format
    lib = L.load()
    fmt = row_format(11, 3)
    ext = lambda f=fmt, sto=16, stride=28 * 10, cap=10, rows=16, n=4, na=3, ctr=16: lib.b2rl_replay_extend_dev_stack(
        sto, stride, cap, f, rows, n, na, ctr, None)
    assert ext(f=L.RowFmt(11, 3, 27, 0)) == -1 and b"row_stride" in lib.b2rl_last_error()  # not a multiple of 4
    for kw in ({"sto": None}, {"rows": None}, {"ctr": None}):
        assert ext(**kw) == -1 and b"non-null" in lib.b2rl_last_error()
    assert ext(sto=8) == -1  # misaligned storage
    assert ext(n=0) == -1 and ext(n=11) == -1  # 1 <= n <= capacity
    assert ext(na=0) == -1 and ext(na=70000) == -1
    assert ext(stride=6) == -1  # not a multiple of 4 floats
    assert ext(stride=28 * 10 - 4) == -1 and b"agent's storage" in lib.b2rl_last_error()  # agents' slices overlap
    assert lib.b2rl_replay_extend_dev(16, 10, fmt, 16, 4, None, None) == -1  # the single-agent form checks the same
    lay = make_layout(11, 3, False, True)
    a = L.UpdateArgs()
    a.hp.td3, a.fmt, a.actor = 0, fmt, lay.actor.c_struct()
    a.arena, a.min_ac, a.max_ac = 16, 16, 16
    a.n_agents, a.agent_base, a.arena_agent_stride = 3, 0, 0
    assert lib.b2rl_actor_predict(C.byref(a), 16, 4, 1, 0.0, C.c_uint64(1), 16, None) == -1  # no agent stride
    assert b"stride" in lib.b2rl_last_error()
    a.arena_agent_stride, a.n_agents = 4 * lay.region, -1
    assert lib.b2rl_actor_predict(C.byref(a), 16, 4, 1, 0.0, C.c_uint64(1), 16, None) == -1
    a.n_agents, a.agent_base = 3, (1 << 30) - 2
    assert lib.b2rl_actor_predict(C.byref(a), 16, 4, 1, 0.0, C.c_uint64(1), 16, None) == -1
