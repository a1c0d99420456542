"""Population-based training over a sharded population: exploit_many moves learner states between global ids with snapshot
semantics (every dst takes its src's state as it was when the round started), on one rank by device copies and between
ranks point to point, bitwise equal to one population that did the same exploits; all_gather puts per-agent values in
global id order on every rank; bad rounds are refused before anything is written. The planning step is checked on the
CPU over random rounds, world sizes 1-8 and uneven shards; the two-rank protocol runs in tests/pbt_worker.py (two ranks
sharing one GPU over gloo, and NCCL on two GPUs). Hopper shapes (O = 11, A = 3), batch 32."""
import os
import random
import subprocess
import sys
from pathlib import Path

import pytest
import torch

REPO = Path(__file__).resolve().parent.parent
ROUND = [(1, 2), (2, 1), (3, 1), (0, 3)]  # a swap (1 <-> 2), 1 read after it was overwritten (3 <- 1), a chain (0 <- 3 <- 1)


# ---- 1. one rank: exploit_many == clone every agent, then copy ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo,wide", [("sac", None), ("td3", None), ("sac", "3xtf32"), ("td3", "3xtf32")])
def test_exploit_many_on_one_rank_equals_clone_then_copy(algo, wide):
    from tests.pbt_worker import assert_same, clone_then_copy, make_pop, state
    pop, ref = make_pop(range(4), algo, wide), make_pop(range(4), algo, wide)
    assert pop.n_total == 4 and [pop.local_index(i) for i in (0, 3, 4)] == [0, 3, None]
    for p in (pop, ref):
        for _ in range(4):
            p.iteration()
    torch.cuda.synchronize()
    assert_same(state(pop), state(ref), "before the round", wide)
    before = state(pop)
    n_graphs = len(pop.graphs)
    pop.exploit_many(ROUND)
    clone_then_copy(ref, ROUND)
    torch.cuda.synchronize()
    got = state(pop)
    assert_same(got, state(ref), f"{algo} {wide}: after the round", wide)
    assert len(pop.graphs) == n_graphs
    assert not torch.equal(got["arena"], before["arena"]) and got["hps"] != before["hps"]  # (the round did something)
    assert torch.equal(got["arena"][0], before["arena"][3]) and got["hps"][2] == before["hps"][1]
    for p in (pop, ref):
        for i in range(4, 7):  # (the same iteration indices: the actor-step cadence follows them)
            p.iteration(i)
    torch.cuda.synchronize()
    assert torch.isfinite(pop.out).all()
    assert_same(state(pop), state(ref), f"{algo} {wide}: 3 iterations after the round", wide)


@pytest.mark.gpu
def test_exploit_many_of_no_pairs_and_of_one_pair_equals_exploit():
    from tests.pbt_worker import assert_same, make_pop, state
    pop, ref = make_pop(range(3), "sac"), make_pop(range(3), "sac")
    for p in (pop, ref):
        p.iteration()
    before = state(pop)
    pop.exploit_many([])
    assert_same(state(pop), before, "no pairs")
    pop.exploit_many([(2, 0)])
    ref.exploit(2, 0)
    torch.cuda.synchronize()
    assert_same(state(pop), state(ref), "one pair")


@pytest.mark.gpu
def test_all_gather_on_one_rank():
    import numpy as np
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from tests.pbt_worker import make_pop
    pop = make_pop(range(3), "sac", use_graphs=False)
    assert np.array_equal(pop.all_gather(torch.arange(3.0, device="cuda")), np.arange(3.0))
    assert pop.all_gather([[1, 2], [3, 4], [5, 6]]).shape == (3, 2)
    with pytest.raises(L.B2rlError, match="one row per local agent"):
        pop.all_gather(np.zeros(4))


@pytest.mark.gpu
def test_bad_rounds_are_refused_before_any_write_on_one_rank():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from tests.pbt_worker import make_pop, state, assert_same
    pop = make_pop(range(4), "sac", wide="3xtf32")
    pop.iteration()
    torch.cuda.synchronize()
    before = state(pop)
    for pairs, msg in [([(4, 0)], r"dst id 4 is outside \[0, n_total = 4\)"), ([(0, -1)], "src id -1 is outside"),
                       ([(1, 0), (2, 3), (1, 3)], "dst 1 appears in more than one pair"),
                       ([(1, 0), (2, 2)], "same agent"), ([(0, 1.0)], "integer global ids"), ([(0,)], "integer global ids"),
                       (5, "integer global ids")]:
        with pytest.raises(L.B2rlError, match=msg):
            pop.exploit_many(pairs)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(L.B2rlError, match="graph capture"):
        with torch.cuda.graph(g):
            pop.exploit_many([(1, 0)])
    torch.cuda.synchronize()
    assert_same(state(pop), before, "after the refusals", "3xtf32")
    # a population that is not the whole id range [0, n_total) has nobody to exploit with
    part = make_pop([2, 3], "sac", use_graphs=False)
    with pytest.raises(L.B2rlError, match="leave a hole"):
        part.exploit_many([(2, 3)])
    with pytest.raises(L.B2rlError, match="leave a hole"):
        part.n_total
    assert part.local_index(3) == 1 and part.local_index(1) is None


# ---- 2. two ranks ---------------------------------------------------------------------------------------------------------------
def _torchrun(port, env, timeout):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(REPO / "tests" / "pbt_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=REPO, env=dict(os.environ, **env))
    print(p.stdout[-3000:], p.stderr[-3000:])
    assert p.returncode == 0 and "PBT_OK" in p.stdout
    assert p.stdout.count("PBT_RESULT") == 4 and "PBT_REFUSALS_OK" in p.stdout


@pytest.mark.gpu
def test_two_rank_pbt_on_one_gpu_over_gloo():
    _torchrun(29541, {"B2RL_PBT_BACKEND": "gloo"}, 900)


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_pbt_over_nccl():
    _torchrun(29542, {}, 900)


# ---- 3. CPU: validation and the plan -------------------------------------------------------------------------------------------
def _random_round(rng, n_total):
    dsts = rng.sample(range(n_total), rng.randint(0, n_total))
    return [(d, rng.choice([s for s in range(n_total) if s != d])) for d in dsts]


def _simulate(pairs, n_total, world):
    """Run every rank's plan on integer states: snapshots first, then copies and transfers with every read of a live row
    checked to be of a row no pair writes (so any order of the writes gives the same result)."""
    from sac_td3_cudagraphs_pytorch_b200.population import plan_exploit, shard
    owner = [r for r in range(world) for _ in shard(n_total, world, r)]
    plans = [plan_exploit(pairs, owner, r) for r in range(world)]
    dsts = {d for d, _ in pairs}
    old = list(range(100, 100 + n_total))
    new = list(old)
    snaps = [{s: old[s] for s in p.snapshots} for p in plans]

    def read(r, s):
        assert owner[s] == r
        if s in snaps[r]:
            return snaps[r][s]
        assert s not in dsts, f"rank {r} reads agent {s}, which this round overwrites, without a snapshot"
        return old[s]
    for r, p in enumerate(plans):
        for d, s in p.copies:
            assert owner[d] == owner[s] == r
            new[d] = read(r, s)
        for peer, d, s in p.sends + p.recvs:
            assert peer != r, f"rank {r} plans a transfer to itself"
    for r, p in enumerate(plans):
        for s_rank in range(world):
            sent = [(d, s) for q, d, s in plans[s_rank].sends if q == r]
            assert sent == [(d, s) for q, d, s in p.recvs if q == s_rank], f"{s_rank} -> {r}: sends != receives"
            for (d, s) in sent:
                assert owner[d] == r and owner[s] == s_rank
                new[d] = read(s_rank, s)
    return old, new


@pytest.mark.parametrize("seed", range(6))
def test_plan_moves_every_src_state_once_over_random_rounds(seed):
    rng = random.Random(seed)
    for _ in range(60):
        n_total, world = rng.randint(2, 40), rng.randint(1, 8)
        pairs = _random_round(rng, n_total)
        old, new = _simulate(pairs, n_total, world)
        want = list(old)
        for d, s in pairs:
            want[d] = old[s]
        assert new == want, (n_total, world, pairs)
        # the order of the pairs does not matter
        assert _simulate(rng.sample(pairs, len(pairs)), n_total, world)[1] == want


def test_plan_of_the_two_rank_round():
    from sac_td3_cudagraphs_pytorch_b200.population import plan_exploit, shard
    from tests.pbt_worker import PAIRS
    owner = [r for r in range(2) for _ in shard(7, 2, r)]
    p0, p1 = plan_exploit(PAIRS, owner, 0), plan_exploit(PAIRS, owner, 1)
    assert p0.copies == [(0, 1), (1, 0)] and p0.snapshots == [0, 1, 2, 3] and p1.copies == [] and p1.snapshots == [4]
    assert p0.sends == [(1, 4, 2), (1, 5, 3)] and p1.recvs == [(0, 4, 2), (0, 5, 3)]
    assert p1.sends == [(0, 2, 4), (0, 3, 6)] and p0.recvs == [(1, 2, 4), (1, 3, 6)]


def test_check_pairs_refuses_bad_rounds():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.population import check_pairs
    import numpy as np
    assert check_pairs([(np.int64(1), 0), (0, 1)], 2) == [(1, 0), (0, 1)]
    assert check_pairs([], 1) == []
    for pairs, msg in [([(2, 0)], "dst id 2 is outside"), ([(0, 5)], "src id 5 is outside"), ([(-1, 0)], "outside"),
                       ([(0, 1), (0, 1)], "dst 0 appears in more than one pair"), ([(1, 1)], "same agent"),
                       ([(0, 1.5)], "integer"), ([("0", 1)], "integer"), ([(0, 1, 2)], "integer"), (None, "integer")]:
        with pytest.raises(L.B2rlError, match=msg):
            check_pairs(pairs, 2)
