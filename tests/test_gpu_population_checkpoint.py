"""Population checkpoints: save / load resume training bitwise on the row path and the 3xTF32 path, across the
environment-facing step, in place (rewinding a population whose graphs are captured) and across a different partition of
the agent ids (re-sharding); per-agent hyperparameters and PBT state survive; the replay may be left out; an exported
member is an Agent checkpoint that trains on exactly as the member does; bad loads are refused before any write.
Hopper shapes (O = 11, A = 3), batch 32 on the row path and 256 / a ragged 200 on the 3xTF32 path."""
import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions

pytestmark = pytest.mark.gpu

OB, AC, CAP = 11, 3, 1000
LO, HI = [-1.0] * AC, [1.0] * AC
REF_TOP_KEYS = {"hps", "timesteps_so_far", "actor", "qnet1", "qnet2", "actor_optimizer", "q_optimizer"}  # agent.py:343-352
NET_KEYS = [f"fc_stack.fc_block_{i}.{m}.{p}" for i in (1, 2) for m in ("fc", "ln") for p in ("weight", "bias")] + \
           ["head.weight", "head.bias"]  # agents/nets.py:66-84
# every value differs between the agents; agent 1 clips, so the population's graphs contain the clipped actor step
SWEEP = {"qnets_lr": [1e-3, 5e-4, 2e-3, 3e-4], "actor_lr": [3e-4, 1e-3, 1e-4, 6e-4], "gamma": [0.99, 0.95, 0.9, 0.999],
         "polyak": [0.005, 0.05, 0.1, 0.02], "clip_norm": [0.0, 0.05, 0.0, 0.0], "targ_ent": [-3.0, -1.0, 0.5, -6.0],
         "td3_std": [0.2, 0.0, 0.4, 0.1], "actor_noise_std": [0.1, 0.3, 0.05, 0.2]}


def _L():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    return L


def _hps(algo, B):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    return (sac_hps if algo == "sac" else td3_hps)(batch_size=B)


def _data(agent_id, n=600):
    return make_synthetic_transitions(n, OB, AC, LO, HI, seed=77 + agent_id)


def _pop(ids, algo, wide=None, B=None, use_graphs=True, agent_hps=None, cap=CAP, n0=600):
    """n0 transitions of each agent's own data in its replay (n0 = 0: an empty replay, for populations that load one)."""
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, OB, AC, LO, HI, _hps(algo, B or (256 if wide else 32)), "cuda", seed=42, rb_capacity=cap,
                     use_graphs=use_graphs, wide=wide, agent_hps=agent_hps)
    if n0:
        for g, aid in enumerate(ids):
            pop.fill_replay(_data(aid, n0), agent=g)
    return pop


def _train(pop, m):
    for _ in range(m):
        pop.iteration()
    torch.cuda.synchronize()


def _state(pops) -> dict:
    """What must be bitwise equal after a resume, rows in the order of the global ids of `pops` (one or a list)."""
    L = _L()
    pops = pops if isinstance(pops, (list, tuple)) else [pops]
    cat = lambda f: torch.cat([f(p) for p in pops]).clone()
    return {"arena P, T, M, V": cat(lambda p: p.arena.flat[:, :L.REGION_G]),
            "counters": cat(lambda p: p.counters[:, [L.CTR_Q, L.CTR_PI, L.CTR_ALPHA, L.CTR_SIZE, L.CTR_CURSOR]]),
            "alpha_state": cat(lambda p: p.alpha_state[:, [0, 2, 3]]), "out": cat(lambda p: p.out), "idx": cat(lambda p: p.idx)}


def _assert_same(a: dict, b: dict):
    for k in a:
        assert torch.equal(a[k], b[k]), f"{k} differs"


# ---- 1. resume ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,wide,B,use_graphs", [("sac", None, 32, True), ("td3", None, 32, True), ("sac", None, 32, False),
                                                    ("sac", "3xtf32", 256, True), ("td3", "3xtf32", 200, True)])
def test_resume_is_bitwise(algo, wide, B, use_graphs, tmp_path):
    ids = [0, 1, 2]
    a = _pop(ids, algo, wide, B, use_graphs)
    _train(a, 5)
    path = a.save(tmp_path / "pop.ckpt")
    assert path == tmp_path / "pop.ckpt" and path.exists() and not (tmp_path / "pop.ckpt.tmp").exists()
    _train(a, 4)
    b = _pop(ids, algo, wide, B, use_graphs, n0=0)
    with torch.no_grad():
        b.arena.flat.mul_(0.5)  # different weights, wrong on purpose
    b.load(path)
    assert (b.iterations, b.size, b.cursor) == (5, 600, 600)
    _train(b, 4)
    assert torch.isfinite(a.out).all()
    _assert_same(_state(a), _state(b))


# ---- 2. the environment-facing step -------------------------------------------------------------------------------------------
def _steps(pop, inputs, finish=True):
    """Pipelined step_async (one step in flight). Returns the log blocks, the actions and the ticket still to be waited for
    (finish=False: the last step is left unwaited)."""
    logs, acts, prev = [], [], None
    for rows, obs in inputs:
        pop.host_rows(rows.shape[1]).copy_(rows)
        pop.host_obs(obs.shape[1]).copy_(obs)
        t = pop.step_async(None, rows.shape[1], n_obs=obs.shape[1])
        acts.append(pop.wait_actions().copy())
        if prev is not None:
            logs.append(pop.wait(prev).clone())
        prev = t
    if finish:
        logs.append(pop.wait(prev).clone())
        torch.cuda.synchronize()
    return logs, acts, prev


@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_step_resumes_bitwise(algo, tmp_path):
    from sac_td3_cudagraphs_pytorch_b200.replay import row_format
    ids, n0, cap, n_new, n_obs = [3, 4, 5], 200, 230, 4, 5  # the cursor wraps after the save point
    gen = torch.Generator().manual_seed(11)
    rs = row_format(OB, AC).row_stride
    inputs = [(torch.randn(len(ids), n_new, rs, generator=gen), torch.randn(len(ids), n_obs, OB, generator=gen))
              for _ in range(14)]
    a = _pop(ids, algo, cap=cap, n0=n0)
    logs, _, last = _steps(a, inputs[:7], finish=False)
    path = a.save(tmp_path / "pop.ckpt")  # with the last step launched and its log block not read yet
    logs.append(a.wait(last).clone())
    assert a.cursor == n0 + 7 * n_new
    want_logs, want_acts, _ = _steps(a, inputs[7:])
    assert a.cursor == (n0 + 14 * n_new) % cap and a.size == cap
    b = _pop(ids, algo, cap=cap, n0=0)
    b.load(path)
    assert (b.size, b.cursor, b.iterations) == (n0 + 7 * n_new, n0 + 7 * n_new, 7)
    got_logs, got_acts, _ = _steps(b, inputs[7:])
    for i in range(7):
        assert torch.equal(got_logs[i], want_logs[i]), f"log block differs at step {7 + i}"
        assert np.array_equal(got_acts[i], want_acts[i]), f"actions differ at step {7 + i}"
    _assert_same(_state(a), _state(b))
    assert torch.equal(a.storage, b.storage) and (a.size, a.cursor) == (b.size, b.cursor)
    # the eager behaviour policy continues its own draws too
    obs = torch.randn(len(ids), 2, OB, generator=gen)
    assert torch.equal(a.predict(obs, explore=True), b.predict(obs, explore=True))


# ---- 3. rewind in place ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,wide", [("sac", None), ("td3", "3xtf32")])
def test_rewind_in_place_keeps_the_captured_graphs(algo, wide, tmp_path):
    ids = [0, 1, 2]
    pop = _pop(ids, algo, wide, B=200 if wide else None)
    if wide:
        pop.lo_mirror()  # a 3xTF32 mirror: load recomputes it from the loaded parameters
    _train(pop, 4)
    path = pop.save(tmp_path / "pop.ckpt")
    _train(pop, 5)
    first = _state(pop)
    graphs = dict(pop.graphs)
    assert graphs
    lo_before = None if pop._lo is None else pop._lo.clone()
    pop.load(path)
    assert pop.iterations == 4
    if wide:
        torch.cuda.synchronize()
        fresh = _pop(ids, algo, wide, B=200, n0=0)
        fresh.load(path)
        assert torch.equal(pop._lo, fresh.lo_mirror()) and not torch.equal(pop._lo, lo_before)
    _train(pop, 5)
    assert pop.graphs == graphs  # no variant was captured again: the same graphs replayed on the loaded state
    _assert_same(first, _state(pop))


# ---- 4. re-sharding -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo,wide,B", [("sac", None, 32), ("td3", "3xtf32", 200)])
def test_checkpoints_reshard(algo, wide, B, tmp_path):
    k, m = 4, 5
    whole = _pop([0, 1, 2, 3], algo, wide, B)
    halves = [_pop([0, 1], algo, wide, B), _pop([2, 3], algo, wide, B)]
    for p in [whole, *halves]:
        _train(p, k)
    f_whole = whole.save(tmp_path / "whole.ckpt")
    f_ranks = [h.save(tmp_path / f"rank{r}.ckpt") for r, h in enumerate(halves)]
    _train(whole, m)
    want = _state(whole)
    # one file of the whole population -> two shards
    shards = [_pop([0, 1], algo, wide, B, n0=0), _pop([2, 3], algo, wide, B, use_graphs=False, n0=0)]
    for s in shards:
        s.load(f_whole)
    # the files of two ranks -> one population, and -> a shard that straddles them (every rank passes every file)
    one = _pop([0, 1, 2, 3], algo, wide, B, n0=0)
    one.load(f_ranks)
    mid = _pop([1, 2], algo, wide, B, n0=0)
    mid.load(f_ranks)
    for p in [*shards, one, mid]:
        _train(p, m)
    _assert_same(want, _state(shards))
    _assert_same(want, _state(one))
    _assert_same({k_: v[1:3] for k_, v in want.items()}, _state(mid))
    assert torch.isfinite(whole.out).all() and not torch.equal(whole.arena.flat[0], whole.arena.flat[1])


# ---- 5. sweeps and PBT state -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_sweep_and_pbt_state_survive(algo, tmp_path):
    ids = [0, 1, 2, 3]
    pop = _pop(ids, algo, agent_hps=SWEEP)
    _train(pop, 3)
    pop.set_agent_hps([1, 2], gamma=0.8, actor_lr=2e-3, targ_ent=-2.0)
    pop.exploit(3, 1)
    pop.set_agent_hps(3, polyak=0.2, clip_norm=0.0)
    _train(pop, 3)
    path = pop.save(tmp_path / "pop.ckpt")
    hp, table = [pop.agent_hps(g) for g in range(4)], pop.agent_hp_table.clone()
    _train(pop, 4)
    b = _pop(ids, algo, agent_hps=SWEEP, n0=0)
    b.load(path)
    assert [b.agent_hps(g) for g in range(4)] == hp
    assert hp[3]["polyak"] == 0.2 and hp[3]["actor_lr"] == 2e-3 and hp[0]["gamma"] == 0.99
    assert torch.equal(b.agent_hp_table, table)
    _train(b, 4)
    _assert_same(_state(pop), _state(b))


# ---- 6. replay left out -----------------------------------------------------------------------------------------------------------
def test_checkpoint_without_replay(tmp_path):
    L = _L()
    ids = [0, 1, 2]
    pop = _pop(ids, "sac")
    _train(pop, 3)
    full, lean = pop.save(tmp_path / "full.ckpt"), pop.save(tmp_path / "lean.ckpt", replay=False)
    assert lean.stat().st_size < full.stat().st_size
    assert "storage" in torch.load(full, mmap=True, weights_only=False)
    assert "storage" not in torch.load(lean, mmap=True, weights_only=False)
    other = _pop(ids, "sac", cap=500, n0=300)  # other data, fill count, cursor and capacity
    before = (other.storage.clone(), other.counters[:, [L.CTR_SIZE, L.CTR_CURSOR]].clone(), other.size, other.cursor)
    other.load(lean)
    torch.cuda.synchronize()
    assert torch.equal(other.storage, before[0]) and torch.equal(other.counters[:, [L.CTR_SIZE, L.CTR_CURSOR]], before[1])
    assert (other.size, other.cursor) == before[2:] == (300, 300)
    assert torch.equal(other.arena.flat[:, :L.REGION_G], pop.arena.flat[:, :L.REGION_G]) and other.iterations == 3
    # with the same data refilled by the caller, training continues bitwise
    again = _pop(ids, "sac")
    again.load(lean)
    _train(pop, 4)
    _train(again, 4)
    _assert_same(_state(pop), _state(again))


# ---- 7. export a member as an Agent checkpoint ---------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_exported_member_is_an_agent_checkpoint(algo, tmp_path):
    from sac_td3_cudagraphs_pytorch_b200 import Hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    L = _L()
    ids, g = [4, 5, 6], 1
    sweep = {"actor_lr": [3e-4, 1e-3, 6e-4], "gamma": [0.99, 0.95, 0.9], "targ_ent": [-3.0, -1.0, 0.5],
             "qnets_lr": [1e-3, 5e-4, 2e-3], "polyak": [0.005, 0.05, 0.1]}
    pop = _pop(ids, algo, agent_hps=sweep)
    _train(pop, 4)
    path = pop.save_agent(g, tmp_path, sfx="best")
    assert path.name == "ckpt_best.pth"
    ck = torch.load(path, weights_only=False)
    assert REF_TOP_KEYS <= set(ck), sorted(ck)
    for k in ("qnet1", "qnet2"):
        assert list(ck[k]) == NET_KEYS
    assert [k for k in ck["actor"] if k.startswith(("fc_stack", "head"))] == NET_KEYS
    assert {"action_scale", "action_bias"} <= set(ck["actor"])
    if algo == "td3":
        assert float(ck["actor"]["exploration_noise"]) == pytest.approx(pop.agent_hps(g)["actor_noise_std"])
    assert ck["qnet1"]["fc_stack.fc_block_1.fc.weight"].shape == (256, OB + AC)
    assert ck["qnet1"]["head.weight"].shape == (1, 256)
    assert ck["qnet_target"]["head.weight"].shape == (2, 1, 256)
    assert ck["q_optimizer"]["state"][0]["exp_avg"].shape == (2, 256, OB + AC)  # stacked like qnet_params
    assert ("alpha_optimizer" in ck) == ("log_alpha" in ck) == (algo == "sac")
    actor_shapes = [v.shape for k, v in ck["actor"].items() if k.startswith(("fc_stack", "head"))]
    stock = torch.optim.Adam([torch.nn.Parameter(torch.zeros(s)) for s in actor_shapes], lr=1.0)
    stock.load_state_dict(ck["actor_optimizer"])
    assert stock.param_groups[0]["lr"] == sweep["actor_lr"][g]
    assert int(stock.state_dict()["state"][0]["step"]) == int(pop.counters[g, L.CTR_PI])
    h = ck["hps"]
    assert (h["actor_lr"], h["gamma"], h["qnets_lr"], h["polyak"], h["targ_ent"]) == tuple(sweep[k][g] for k in (
        "actor_lr", "gamma", "qnets_lr", "polyak", "targ_ent"))
    assert h["batch_size"] == pop.hps.batch_size
    assert "targ_ent" not in torch.load(pop.save_agent(0, tmp_path, sfx="m0"), weights_only=False)["hps"]  # -A: no key

    aid = pop.base + g
    rb = ReplayBuffer(CAP, "cuda", seed=pop.seed, agent_id=aid)
    rb.extend({k: v.cuda() for k, v in _data(aid).items()})
    ag = Agent({"ob_shape": (OB,), "ac_shape": (AC,)}, np.array(LO), np.array(HI), torch.device("cuda"), Hps(ck["hps"]),
               rb=rb, seed=pop.seed, agent_id=aid)
    ag.load_from_disk(path)
    torch.cuda.synchronize()
    for r in range(4):
        assert torch.equal(ag.arena.flat[0, r], pop.arena.flat[g, r]), f"region {r}"
    assert torch.equal(ag.counters[:3], pop.counters[g, :3])
    if algo == "sac":
        assert torch.equal(ag._alpha_state[[0, 2, 3]], pop.alpha_state[g, [0, 2, 3]])
        assert ag.targ_ent == -1.0
    eng = LearnerEngine(ag, use_graphs=False)
    ag.qnet_updates_so_far = pop.iterations
    for i in range(pop.iterations, pop.iterations + 6):
        pop.iteration()
        eng.iteration(i)
    torch.cuda.synchronize()
    assert torch.equal(pop.arena.flat[g], ag.arena.flat[0]), "exported agent != member"
    assert torch.equal(pop.counters[g, :3], ag.counters[:3])
    assert torch.equal(pop.alpha_state[g, :4], ag._alpha_state[:4])
    assert torch.equal(pop.out[g, :4], ag.out[:4])


# ---- 8. refusals ---------------------------------------------------------------------------------------------------------------
def test_bad_loads_and_calls_are_refused(tmp_path):
    L = _L()
    ids = [0, 1, 2, 3]
    src = _pop(ids, "sac")
    _train(src, 2)
    path = src.save(tmp_path / "pop.ckpt")
    target = _pop(ids, "sac")
    _train(target, 1)
    snap = {k: getattr(target, k).clone() for k in ("storage", "counters", "alpha_state", "agent_hp_table")}
    snap["arena"] = target.arena.flat.clone()
    host = (target.size, target.cursor, target.iterations, target.agent_hps(0))

    def variant(name, edit):
        ck = torch.load(path, weights_only=False)
        edit(ck)
        p = tmp_path / name
        torch.save(ck, p)
        return p

    (tmp_path / "junk").write_bytes(b"not a checkpoint")
    torch.save({"hps": {}, "actor": {}}, tmp_path / "agent.pth")
    cases = [
        (tmp_path / "junk", "format"),
        (tmp_path / "agent.pth", "format"),
        (variant("v2", lambda c: c.update(version=2)), "version"),
        (variant("algo", lambda c: c["hps"].update(prefer_td3_over_sac=True)), "prefer_td3_over_sac"),
        (variant("ob", lambda c: c.update(ob_dim=OB + 1)), "ob_dim"),
        (variant("ac", lambda c: c.update(ac_dim=AC + 1)), "ac_dim"),
        (variant("ln", lambda c: c["hps"].update(layer_norm=False)), "layer_norm"),
        (variant("lo", lambda c: c.update(min_ac=[-2.0] * AC)), "min_ac"),
        (variant("hi", lambda c: c.update(max_ac=[2.0] * AC)), "max_ac"),
        (variant("region", lambda c: c.update(region=c["region"] + 4)), "region"),
        (variant("stride", lambda c: c.update(row_stride=32)), "row_stride"),
        (variant("seed", lambda c: c.update(seed=43)), "seed"),
        (variant("cap", lambda c: c.update(capacity=2 * CAP)), "capacity"),
        (_pop([0, 1], "sac", n0=0).save(tmp_path / "two.ckpt"), "ids: agent 2 is in none"),
        ([path, path], "more than one"),
        (_pop(ids, "sac", agent_hps={"clip_norm": [0.0, 0.1, 0.0, 0.0]}, n0=0).save(tmp_path / "clip.ckpt"), "clip_norm"),
        (_pop(ids, "sac", n0=0, agent_hps={"log_alpha_lr": [0.0] * 4}).save(tmp_path / "noalpha.ckpt"), "log_alpha_lr"),
    ]
    for p, msg in cases:
        with pytest.raises(L.B2rlError, match=msg):
            target.load(p)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        with pytest.raises(L.B2rlError, match="capture"):
            target.load(path)
        with pytest.raises(L.B2rlError, match="capture"):
            target.save(tmp_path / "in_capture.ckpt")
    assert not (tmp_path / "in_capture.ckpt").exists()
    torch.cuda.synchronize()
    for k, v in snap.items():
        assert torch.equal(v, target.arena.flat if k == "arena" else getattr(target, k)), f"a refused load changed {k}"
    assert (target.size, target.cursor, target.iterations, target.agent_hps(0)) == host
    # without the replay, another capacity is fine
    target.load(_pop(ids, "sac", cap=500, n0=0).save(tmp_path / "lean.ckpt", replay=False))
    assert target.capacity == CAP and target.size == host[0]
