"""torchrun worker for tests/test_gpu_population_pbt.py: population-based training over a population sharded on W ranks
(exploit_many, all_gather) equals a one-rank population of the same global ids that did the same exploits, bitwise;
bad rounds are refused on every rank before anything is written. Also the helpers the one-rank tests share."""
import os
import sys
from datetime import timedelta
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import make_synthetic_transitions  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200 import _lib as L, sac_hps, td3_hps  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.population import Population, shard  # noqa: E402

OB, AC, B, CAP = 11, 3, 32, 1000
N_TOTAL = 7
# every agent has its own values; agents 1 and 5 clip, so every population's graphs contain the clipped actor step
SWEEP = {"qnets_lr": [1e-3, 5e-4, 2e-3, 3e-4, 8e-4, 1.5e-3, 6e-4], "actor_lr": [3e-4, 1e-3, 1e-4, 6e-4, 2e-4, 5e-4, 8e-4],
         "gamma": [0.99, 0.95, 0.9, 0.999, 0.97, 0.98, 0.93], "polyak": [0.005, 0.05, 0.1, 0.02, 0.01, 0.03, 0.07],
         "td3_std": [0.2, 0.0, 0.4, 0.1, 0.3, 0.15, 0.25], "actor_noise_std": [0.1, 0.3, 0.05, 0.2, 0.15, 0.25, 0.12],
         "alpha_init": [0.2, 0.5, 0.05, 1.0, 0.3, 0.1, 0.7], "targ_ent": [-3.0, -1.0, 0.5, -6.0, -2.0, -4.0, -1.5],
         "clip_norm": [0.0, 0.05, 0.0, 0.0, 0.0, 0.02, 0.0]}
WIDE_SWEEP = dict(SWEEP, clip_norm=[0.0] * N_TOTAL)  # (the tensor-core actor step has no gradient clipping)
# one round with every kind of pair over shard(7, 2, .) = [0, 4) + [4, 7): a swap on rank 0 (0 <-> 1), a swap across ranks
# (2 <-> 4), a chain across ranks (6 -> 3 -> 5: 3 is a dst on rank 0 and the src of a dst on rank 1)
PAIRS = [(1, 0), (0, 1), (4, 2), (2, 4), (3, 6), (5, 3)]
PATHS = [("sac", None), ("td3", None), ("sac", "3xtf32"), ("td3", "3xtf32")]


def sweep_of(ids, wide, sweep=None):
    sweep = sweep or (WIDE_SWEEP if wide else SWEEP)
    return {k: [v[i] for i in ids] for k, v in sweep.items()}


def make_pop(ids, algo, wide=None, sweep=None, use_graphs=True, **over):
    ids = list(ids)
    hps = (sac_hps if algo == "sac" else td3_hps)(batch_size=B, **over)
    pop = Population(ids, OB, AC, [-1.0] * AC, [1.0] * AC, hps, "cuda", seed=42, rb_capacity=CAP, use_graphs=use_graphs,
                     wide=wide, agent_hps=sweep_of(ids, wide, sweep))
    for g, aid in enumerate(ids):
        pop.fill_replay(make_synthetic_transitions(600, OB, AC, [-1.0] * AC, [1.0] * AC, seed=77 + aid), agent=g)
    if wide:
        pop.lo_mirror()  # (kept by the optimizer launches; exploit_many moves or rebuilds its rows too)
    return pop


def state(pop, rows=slice(None)) -> dict:
    """Everything a PBT round may change or must keep, for local agents `rows`; host hyperparameters as a list."""
    st = {"arena": pop.arena.flat[rows], "alpha_state": pop.alpha_state[rows], "counters": pop.counters[rows],
          "out": pop.out[rows], "agent_hp_table": pop.agent_hp_table[rows], "storage": pop.storage[rows]}
    if pop._lo is not None:
        st["lo"] = pop._lo[rows]
    st = {k: v.clone() for k, v in st.items()}
    st["hps"] = [pop.agent_hps(g) for g in range(pop.N)[rows]]
    return st


def assert_same(a: dict, b: dict, what: str, wide=None):
    assert a.keys() == b.keys(), (what, a.keys(), b.keys())
    for k in a:
        x, y = a[k], b[k]
        if k == "alpha_state" and wide:  # log alpha and its Adam moments, as the other population tests compare the wide path
            x, y = x[:, [0, 2, 3]], y[:, [0, 2, 3]]
        assert (x == y) if k == "hps" else torch.equal(x, y), f"{what}: {k} differs"


def clone_then_copy(pop, pairs):
    """The meaning of exploit_many on one rank: clone every agent's state, then let each dst take its src's clone."""
    torch.cuda.synchronize()
    old = state(pop)
    with torch.no_grad():
        for d, s in pairs:
            pop.arena.flat[d].copy_(old["arena"][s])
            pop.alpha_state[d].copy_(old["alpha_state"][s])
            pop.counters[d, L.CTR_Q:L.CTR_ALPHA + 1].copy_(old["counters"][s, L.CTR_Q:L.CTR_ALPHA + 1])
            pop.agent_hp_table[d].copy_(old["agent_hp_table"][s])
            if pop._lo is not None:
                pop._lo[d].copy_(old["lo"][s])
            pop._hp[d] = dict(old["hps"][s])


def step_inputs(n_agents, n_it, n_new=4, n_obs=4, seed=3):
    rs = pop_row_stride()
    gen = torch.Generator().manual_seed(seed)
    return [(torch.randn(n_agents, n_new, rs, generator=gen), torch.randn(n_agents, n_obs, OB, generator=gen))
            for _ in range(n_it)]


def pop_row_stride():
    from sac_td3_cudagraphs_pytorch_b200.replay import row_format
    return row_format(OB, AC).row_stride


def run_steps(pop, inputs):
    for rows, obs in inputs:
        pop.host_rows(rows.shape[1]).copy_(rows)
        pop.host_obs(obs.shape[1]).copy_(obs)
        pop.wait(pop.step_async(None, rows.shape[1], n_obs=obs.shape[1]))


def perturb(pop, dsts, seed=11):
    """The explore half, from an RNG seeded the same everywhere: every rank draws for every dst, applies its own."""
    rng = np.random.default_rng(seed)
    for d in dsts:
        f = rng.choice([0.8, 1.25])
        g = pop.local_index(d)
        if g is not None:
            h = pop.agent_hps(g)
            pop.set_agent_hps(g, qnets_lr=h["qnets_lr"] * f, gamma=min(0.999, h["gamma"] * 1.005))


def train_after_round(pop, inputs):
    """4 steps through the step graph, then 2 iterations on the eager path."""
    run_steps(pop, inputs)
    pop.use_graphs = False
    for _ in range(2):
        pop.iteration()
    pop.use_graphs = True
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- workers
def sharded_equals_one_rank(rank, world, solo):
    mine = shard(N_TOTAL, world, rank)
    inputs = step_inputs(N_TOTAL, 4)
    for algo, wide in PATHS:
        pop = make_pop(mine, algo, wide)
        ref = make_pop(range(N_TOTAL), algo, wide)
        assert pop.n_total == N_TOTAL and ref._ranks(solo).n_total == N_TOTAL
        for p in (pop, ref):
            for _ in range(4):
                p.iteration()
        torch.cuda.synchronize()
        before = state(pop)
        pop.exploit_many(PAIRS)
        ref.exploit_many(PAIRS, group=solo)
        torch.cuda.synchronize()
        after = state(pop)
        # dsts keep their replay slices, replay counters and log blocks
        assert torch.equal(after["storage"], before["storage"])
        assert torch.equal(after["counters"][:, L.CTR_SAMPLE:], before["counters"][:, L.CTR_SAMPLE:])
        assert torch.equal(after["out"], before["out"])
        assert_same(after, state(ref, slice(mine.start, mine.stop)), f"{algo} {wide} rank {rank} after the round", wide)
        dsts = [d for d, _ in PAIRS]
        perturb(pop, dsts)
        perturb(ref, dsts)
        train_after_round(pop, [(r[mine.start:mine.stop], o[mine.start:mine.stop]) for r, o in inputs])
        train_after_round(ref, inputs)
        assert_same(state(pop), state(ref, slice(mine.start, mine.stop)), f"{algo} {wide} rank {rank} after training", wide)
        assert torch.isfinite(pop.out).all()
        # every rank ranks the same gathered scores
        scores = pop.all_gather(pop.out[:, L.OUT_QF_LOSS])
        assert scores.shape == (N_TOTAL,) and np.array_equal(scores, ref.out[:, L.OUT_QF_LOSS].cpu().numpy())
        everyone = [None] * world
        dist.all_gather_object(everyone, scores)
        assert all(np.array_equal(s, scores) for s in everyone)
        two = pop.all_gather(np.stack([np.arange(len(mine)) + mine.start] * 2, 1))
        assert np.array_equal(two, np.stack([np.arange(N_TOTAL)] * 2, 1))
        if rank == 0:
            print(f"PBT_RESULT {algo} wide={wide} world={world} bitwise", flush=True)


def expect_refusal(pops, call, match, what):
    """call() must raise a B2rlError naming `match` on this rank and change none of `pops`."""
    torch.cuda.synchronize()
    before = [state(p) for p in pops]
    try:
        call()
    except L.B2rlError as e:
        assert match in str(e), f"{what}: {e}"
    else:
        raise AssertionError(f"{what}: not refused")
    torch.cuda.synchronize()
    for p, b in zip(pops, before):
        assert_same(state(p), b, what)


def refusals(rank, world):
    mine = shard(N_TOTAL, world, rank)
    pop = make_pop(mine, "sac", use_graphs=False)
    pop.iteration()
    expect_refusal([pop], lambda: pop.exploit_many([(N_TOTAL, 0)]), "outside [0, n_total = 7)", "id out of range")
    expect_refusal([pop], lambda: pop.exploit_many([(-1, 0)]), "outside", "negative id")
    expect_refusal([pop], lambda: pop.exploit_many([(1, 4), (1, 5)]), "dst 1 appears in more than one pair", "duplicate dst")
    expect_refusal([pop], lambda: pop.exploit_many([(5, 5)]), "the same agent", "dst == src")
    expect_refusal([pop], lambda: pop.exploit_many([(0, 4 + rank)]), "pair lists differ", "pair lists differ")
    expect_refusal([pop], lambda: pop.exploit_many([(0, "a")] if rank == 1 else [(0, 4)]), "integer global ids",
                   "a malformed pair list on one rank")
    # a src that clips cannot go to a population whose graphs have no clipped step
    other = make_pop(mine, "sac", use_graphs=False, sweep=dict(SWEEP, clip_norm=[0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0])
                     if rank == world - 1 else None)
    expect_refusal([other], lambda: other.exploit_many([(N_TOTAL - 1, 1)]), "clipped actor step", "graph variant")
    # configurations that differ between ranks, and id ranges that overlap or leave a hole
    bad = make_pop(mine, "td3" if rank == world - 1 else "sac", use_graphs=False)
    expect_refusal([bad], lambda: bad.exploit_many([(0, 4)]), "configurations differ", "algorithm differs")
    bad = make_pop(mine, "sac", use_graphs=False, layer_norm=rank == 0)
    expect_refusal([bad], lambda: bad.exploit_many([(0, 4)]), "layer_norm", "layer_norm differs")
    over = make_pop(range(mine.start, mine.stop + 1) if rank < world - 1 else mine, "sac", use_graphs=False)
    expect_refusal([over], lambda: over.exploit_many([(0, 4)]), "overlap", "overlapping ids")
    hole = make_pop(range(mine.start, mine.stop - 1) if rank == 0 else mine, "sac", use_graphs=False)
    expect_refusal([hole], lambda: hole.exploit_many([(0, 4)]), "leave a hole", "a hole in the ids")
    expect_refusal([hole], lambda: hole.all_gather(np.zeros(hole.N)), "leave a hole", "a hole in the ids (all_gather)")
    # and a good round still works on the population the refusals were tried on
    pop.exploit_many([(0, 4), (4, 0)])
    if rank == 0:
        print(f"PBT_REFUSALS_OK world={world}", flush=True)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    # B2RL_PBT_BACKEND=gloo: the ranks share GPU 0 and transfer through host buffers (NCCL refuses two ranks on one device)
    backend = os.environ.get("B2RL_PBT_BACKEND", "nccl")
    local = local % torch.cuda.device_count() if backend == "gloo" else local
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    timeout = timedelta(seconds=120)  # a rank left waiting in a collective fails the run instead of hanging it
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev, timeout=timeout)
    else:
        dist.init_process_group("gloo", timeout=timeout)
    solo = [dist.new_group([r]) for r in range(world)][rank]  # a one-rank group: the reference population of all 7 ids
    sharded_equals_one_rank(rank, world, solo)
    refusals(rank, world)
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0:
        print("PBT_OK", flush=True)


if __name__ == "__main__":
    main()
