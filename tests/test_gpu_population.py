"""Population (BASELINE.json config 4): N stacked learners == N separate learners, bitwise, and the result
does not depend on how the agent ids are sharded (the multi-GPU story: a partition, no collective)."""
import numpy as np
import pytest
import torch

from oracle import make_synthetic_transitions

pytestmark = pytest.mark.gpu


def _hps(algo):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    return (sac_hps if algo == "sac" else td3_hps)(batch_size=32)


def _data(agent_id, n=600, ob=11, ac=3):
    return make_synthetic_transitions(n, ob, ac, [-1.0] * ac, [1.0] * ac, seed=77 + agent_id)


def _population(ids, algo, use_graphs=True):
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    pop = Population(ids, 11, 3, [-1.0] * 3, [1.0] * 3, _hps(algo), "cuda", seed=42, rb_capacity=1000,
                     use_graphs=use_graphs)
    for g, aid in enumerate(ids):
        pop.fill_replay(_data(aid), agent=g)
    return pop


@pytest.mark.parametrize("algo", ["sac", "td3"])
def test_population_equals_separate_agents(algo):
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.population import init_agent_params
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    ids, n_it = [5, 6, 7], 7
    pop = _population(ids, algo)
    for i in range(n_it):
        pop.iteration()
    torch.cuda.synchronize()
    hps = _hps(algo)
    lo, hi = torch.full((3,), -1.0), torch.full((3,), 1.0)
    for g, aid in enumerate(ids):
        rb = ReplayBuffer(1000, "cuda", seed=42, agent_id=aid)
        rb.extend({k: v.cuda() for k, v in _data(aid).items()})
        ag = Agent({"ob_shape": (11,), "ac_shape": (3,)}, lo.numpy(), hi.numpy(), torch.device("cuda"), hps, rb=rb,
                   seed=42, agent_id=aid)
        ag.load_params(*init_agent_params(aid, 42, 11, 3, algo == "td3", True, lo, hi))
        eng = LearnerEngine(ag, use_graphs=False)
        for i in range(n_it):
            eng.iteration(i)
        torch.cuda.synchronize()
        assert torch.equal(pop.arena.flat[g], ag.arena.flat[0]), f"agent {aid}: stacked != separate"
        assert torch.equal(pop.counters[g, :3], ag.counters[:3])
        assert torch.equal(pop.alpha_state[g, :4], ag._alpha_state[:4])
        assert torch.equal(pop.out[g, :4], ag.out[:4])
    # agents are independent: different data and seeds give different parameters
    assert not torch.equal(pop.arena.flat[0], pop.arena.flat[1])
    assert torch.isfinite(pop.out).all()


def test_population_is_invariant_to_sharding():
    whole = _population([0, 1, 2, 3], "sac")
    parts = [_population([0, 1], "sac"), _population([2, 3], "sac", use_graphs=False)]
    for i in range(6):
        whole.iteration()
        for p in parts:
            p.iteration()
    torch.cuda.synchronize()
    got = torch.cat([p.arena.flat for p in parts])
    assert torch.equal(whole.arena.flat, got)
    assert torch.equal(whole.idx, torch.cat([p.idx for p in parts]))  # same index draws per global agent id


# ---- the population on the tensor-core (wide) path: agents stacked along the rows ----------------------------------------------
def _wide_population(ids, algo, B, use_graphs=True, wide="3xtf32"):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    hps = (sac_hps if algo == "sac" else td3_hps)(batch_size=B)
    pop = Population(ids, 11, 3, [-1.0] * 3, [1.0] * 3, hps, "cuda", seed=42, rb_capacity=1000, use_graphs=use_graphs, wide=wide)
    for g, aid in enumerate(ids):
        pop.fill_replay(_data(aid), agent=g)
    return pop


@pytest.mark.parametrize("algo,B", [("sac", 256), ("td3", 200)])
def test_wide_population_is_invariant_to_sharding(algo, B):
    """Bitwise: [0,1,2,3] on one GPU == [0,1] + [2] + [3] (graph replay and eager launches) — the multi-GPU contract of
    BASELINE.json config 4 (a partition of the agent ids, no collective) on the tcgen05 path. B = 200 is ragged against
    the 128-row tiles: an agent's tail rows are zero-filled by TMA, never read from its neighbour."""
    whole = _wide_population([0, 1, 2, 3], algo, B)
    parts = [_wide_population([0, 1], algo, B), _wide_population([2], algo, B, use_graphs=False), _wide_population([3], algo, B)]
    for i in range(7):
        whole.iteration()
        for p in parts:
            p.iteration()
    torch.cuda.synchronize()
    assert torch.isfinite(whole.out).all()
    assert torch.equal(whole.arena.flat, torch.cat([p.arena.flat for p in parts]))
    assert torch.equal(whole.counters[:, :3], torch.cat([p.counters[:, :3] for p in parts]))
    assert torch.equal(whole.out, torch.cat([p.out for p in parts]))
    assert torch.equal(whole.alpha_state[:, [0, 2, 3]], torch.cat([p.alpha_state[:, [0, 2, 3]] for p in parts]))
    assert not torch.equal(whole.arena.flat[0], whole.arena.flat[1])


@pytest.mark.parametrize("algo,B", [("sac", 256), ("td3", 256), ("sac", 1000), ("td3", 1000)],
                         ids=["sac", "td3", "sac-1000", "td3-1000"])
def test_wide_population_matches_the_fp32_row_path(algo, B):
    """Same agents, data, index draws and noise on the row-group fp32 kernels and on the stacked 3xTF32 tensor-core path:
    after the first iteration (critic step + two actor steps from identical state) the losses agree to 2e-5, the critics'
    gradients to 5e-5 of each agent's largest entry (stated 3xTF32 bound; a ReLU unit within ~1e-6 of its kink may flip
    between two correct evaluations — seeds are fixed, and none does here), and after 6 iterations the parameters to 2e-3
    (Adam's first steps move every weight by lr whatever the gradient's size, which amplifies rounding-level differences).
    B = 1000 gives every agent several CTAs of each wide kernel (8 tiles of 128 rows, 4 of 256, 125 head groups of 8) and a
    ragged last tile, with the agents' rows stacked back to back."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    ids = [3, 4, 5]
    wide, row = _wide_population(ids, algo, B), _wide_population(ids, algo, B, wide=None)
    wide.iteration()
    row.iteration()
    torch.cuda.synchronize()
    assert torch.equal(wide.idx, row.idx)
    lay = wide.layout
    for g in range(len(ids)):
        for k in (L.OUT_QF_LOSS, L.OUT_ACTOR_LOSS):
            a, b = float(wide.out[g, k]), float(row.out[g, k])
            assert abs(a - b) <= 2e-5 * max(abs(b), 1e-3), (g, k, a, b)
        if algo == "sac":
            # The temperature step draws its own noise (stream 3, keyed on the actor counter after the actor step advanced
            # it), so it checks that key on the wide path. Its loss alpha * (mean(-logpi) - targ_ent) is a difference of
            # O(A) terms, judged against alpha * A (helpers.alpha_loss_scale). A draw keyed on another counter moves
            # mean(-logpi) by ~sqrt(A / 2B) ~ 0.08, i.e. ~3e-2 of that scale. Measured on a B200: <= 5e-7 of alpha * A, and
            # log alpha equal after the two Adam steps.
            a, b = float(wide.out[g, L.OUT_ALPHA_LOSS]), float(row.out[g, L.OUT_ALPHA_LOSS])
            sc = float(row.out[g, L.OUT_ALPHA]) * 3
            la_w, la_r = float(wide.alpha_state[g, 0]), float(row.alpha_state[g, 0])
            print(f"agent {ids[g]}: alpha loss wide {a:.7f} row {b:.7f} (|d| / alpha A = {abs(a - b) / sc:.2e}), "
                  f"log alpha |d| {abs(la_w - la_r):.2e}")
            assert abs(a - b) <= 1e-4 * sc, (g, a, b)
            assert abs(la_w - la_r) <= 1e-6, (g, la_w, la_r)
        for c in lay.critic:  # (the reference's tensors: the w2n shadow has no gradient of its own on the wide path)
            gw = wide.arena.flat[g, L.REGION_G, c.begin:c.core_end]
            gr = row.arena.flat[g, L.REGION_G, c.begin:c.core_end]
            d = float((gw - gr).abs().max()) / float(gr.abs().max())
            assert d <= 5e-5, f"agent {ids[g]}: critic gradients differ by {d:.2e}"
    for i in range(5):
        wide.iteration()
        row.iteration()
    torch.cuda.synchronize()
    for r in (L.REGION_P, L.REGION_T):
        pw, pr = wide.arena.flat[:, r], row.arena.flat[:, r]
        d = float((pw - pr).abs().max()) / float(pr.abs().max())
        assert d <= 2e-3, f"region {r}: parameters differ by {d:.2e} after 6 iterations"
    assert torch.equal(wide.counters[:, :3], row.counters[:, :3])
