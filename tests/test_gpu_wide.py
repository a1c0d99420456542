"""The wide (tensor-core) critic update vs the fp32 oracle and vs the row-group path, same state and noise.
Stated tolerance: TF32 products in the 256x256 hidden layers (forward and dX) — 5e-3 of each tensor's max for
losses / Q values / gradients; parameters after the Adam step get the first-step bound with that tolerance."""
import pytest
import torch

from tests.golden.cases import CASES, case_inputs
from tests.helpers import batch_of, kink_safe, kink_safe_actor, make_agent, make_oracle, rel_dev

pytestmark = pytest.mark.gpu


# (Q / TD target / loss, gradients). tf32: dLoss/dQ = 2 (q - y) / B is a DIFFERENCE of two TF32-accurate values, so the
# 1e-3 of the products becomes ~1e-2 of the TD error and of everything back-propagated from it (more without LayerNorm,
# whose scale invariance absorbs the truncation bias). 3xtf32: the fp32 path's bound.
TOLS = {"3xtf32": (1e-5, 2e-5), "tf32": (5e-3, 1.5e-1)}


@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("name", ["sac_hopper", "td3_hopper", "sac_humanoid", "sac_noln_fixedalpha_bcq", "td3_ant_mixed_first"])
def test_wide_critic_step_matches_oracle(name, precision):
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    from sac_td3_cudagraphs_pytorch_b200.wide import WideCritic
    inp = case_inputs(name)
    ag = make_agent(inp)
    o32 = make_oracle(inp, torch.float32)
    batch = batch_of(inp, 0)
    keep = kink_safe(inp, batch)
    batch = {k: v[keep] for k, v in batch.items()}
    eps = inp["eps_q"][0][keep].contiguous()
    B = int(keep.sum())
    assert B >= 0.75 * inp["B"], "the kink filter should only drop a few rows"
    rows = pack_rows({k: v.cuda() for k, v in batch.items()}, ag.fmt)
    wc = WideCritic(ag, B, precision)
    TOL, GTOL = TOLS[precision]
    tq = torch.zeros(B, device="cuda")
    out = wc.update_qnets(rows, eps=eps.cuda(), targ_out=tq)
    r32 = o32.update_qnets(batch, eps)
    torch.cuda.synchronize()
    assert rel_dev(tq, r32["_targ_q"]) <= TOL
    assert rel_dev(wc.q, r32["_q"].reshape(2, B)) <= TOL
    assert rel_dev(out["loss/qf_loss"], r32["loss/qf_loss"]) <= TOL
    worst = 0.0
    for n, p in ag.qnet_params.items():
        d = rel_dev(p.grad, o32.qnet[n].grad)
        worst = max(worst, d)
        assert d <= GTOL, f"grad {n}: {d:.3e}"
    print(f"\n[{name}] wide critic ({precision}, B={B}) vs fp32 oracle: worst gradient deviation {worst:.2e}")
    for k, q in enumerate((ag.qnet1, ag.qnet2)):  # the natural-layout shadow stays identical to the primary copy
        w = q.fc_stack.fc_block_2.fc.weight.detach()
        assert torch.equal(ag.arena.tensor(ag.layout.critic[k], "w2n"), w.contiguous())
    assert int(ag.counters[0]) == 1


@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("name", ["sac_hopper", "td3_hopper", "sac_humanoid", "sac_noln_fixedalpha_bcq", "td3_ant_mixed_first"])
def test_wide_actor_step_matches_oracle(name, precision):
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    from sac_td3_cudagraphs_pytorch_b200.wide import WideActor
    from tests.helpers import alpha_loss_scale
    inp = case_inputs(name)
    ag = make_agent(inp)
    o32 = make_oracle(inp, torch.float32)
    batch = batch_of(inp, 0)
    e1, e2 = inp["eps_pi"][0][0], inp["eps_alpha"][0][0]
    keep = kink_safe_actor(inp, batch, e1)
    batch = {k: v[keep] for k, v in batch.items()}
    e1, e2 = e1[keep].contiguous(), e2[keep].contiguous()
    B = int(keep.sum())
    assert B >= 0.75 * inp["B"]
    rows = pack_rows({k: v.cuda() for k, v in batch.items()}, ag.fmt)
    wa = WideActor(ag, B, precision)
    TOL, GTOL = TOLS[precision]
    out = wa.update_actor(rows, eps=e1.cuda(), eps_alpha=e2.cuda())
    r32 = o32.update_actor(batch, e1, e2)
    torch.cuda.synchronize()
    for k in r32:
        sc = alpha_loss_scale(inp["hps"]["alpha_init"], inp["ac"]) if k == "loss/alpha_loss" else None
        d = rel_dev(out[k], r32[k], sc)
        assert d <= 10 * TOL, f"{k}: {d:.3e}"
    worst = 0.0
    for n, p in ag.actor_params.items():
        d = rel_dev(p.grad, o32.actor[n].grad)
        worst = max(worst, d)
        assert d <= GTOL, f"grad {n}: {d:.3e}"
    print(f"\n[{name}] wide actor ({precision}, B={B}) vs fp32 oracle: worst gradient deviation {worst:.2e}")
    if not ag.td3 and ag.autotune:
        assert rel_dev(ag.log_alpha, o32.log_alpha) <= 1e-5
    assert int(ag.counters[1]) == 1


@pytest.mark.parametrize("name,wide", [("sac_hopper", "3xtf32"), ("td3_hopper", "3xtf32"), ("sac_hopper", None)])
def test_dp_learner_graph_replay_equals_eager(name, wide):
    """One-rank DataParallelLearner: the captured iteration graphs (one per variant: actor updates? Polyak?) replay the
    same launches as the eager loop — parameters, optimizer state and counters bitwise equal after 9 iterations
    (the first occurrence of every variant runs eagerly, the second is captured and replayed, later ones replay)."""
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    from sac_td3_cudagraphs_pytorch_b200.dp import DataParallelLearner, GradComm
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs(name)
    agents, dps = [], []
    for graphs in (True, False):
        ag = make_agent(inp, seed=5)
        rb = ReplayBuffer(300, "cuda", seed=5)
        rb.extend({k: v[:250].cuda() for k, v in inp["storage"].items()})
        agents.append(ag)
        dps.append(DataParallelLearner(ag, rb, 200, GradComm(), wide=wide, graphs=graphs))
    for i in range(9):
        for dp in dps:
            dp.iteration(i)
    torch.cuda.synchronize()
    assert len(dps[0]._graphs) >= 2 and not dps[1]._graphs
    assert torch.equal(agents[0].arena.flat, agents[1].arena.flat)
    assert torch.equal(agents[0].counters[:4], agents[1].counters[:4])
    assert torch.equal(agents[0].out, agents[1].out)
    assert agents[0].qnet_updates_so_far == agents[1].qnet_updates_so_far == 9
    assert agents[0].actor_updates_so_far == agents[1].actor_updates_so_far


@pytest.mark.parametrize("name", ["sac_hopper", "td3_hopper", "sac_humanoid", "sac_noln_fixedalpha_bcq", "td3_ant_mixed_first"])
def test_wide_critic_step_bound_on_the_whole_batch(name):
    """The same comparison WITHOUT the kink filter (every row of the fixture batch): forward quantities — Q, TD target,
    loss — keep the 1e-5 bound (a unit that flips sits within ~1e-6 of zero, so its activation moves by that much);
    gradients get the stated kink-inclusive bound of 3e-2 of each tensor's max (one flipped unit of one row moves its
    row of the weight gradient by O(1/B); measured worst: printed, 1.0e-2 on td3_hopper)."""
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    from sac_td3_cudagraphs_pytorch_b200.wide import WideCritic
    inp = case_inputs(name)
    ag = make_agent(inp)
    o32 = make_oracle(inp, torch.float32)
    batch = batch_of(inp, 0)
    B = inp["B"]
    rows = pack_rows({k: v.cuda() for k, v in batch.items()}, ag.fmt)
    wc = WideCritic(ag, B, "3xtf32")
    tq = torch.zeros(B, device="cuda")
    out = wc.update_qnets(rows, eps=inp["eps_q"][0].cuda(), targ_out=tq)
    r32 = o32.update_qnets(batch, inp["eps_q"][0])
    torch.cuda.synchronize()
    assert rel_dev(tq, r32["_targ_q"]) <= 1e-5
    assert rel_dev(wc.q, r32["_q"].reshape(2, B)) <= 1e-5
    assert rel_dev(out["loss/qf_loss"], r32["loss/qf_loss"]) <= 1e-5
    devs = {n: rel_dev(p.grad, o32.qnet[n].grad) for n, p in ag.qnet_params.items()}
    worst = max(devs.values())
    print(f"\n[{name}] wide critic, whole batch (B={B}): worst gradient deviation {worst:.2e}; tensors above 2e-5: "
          f"{[n for n, d in devs.items() if d > 2e-5]}")
    assert worst <= 3e-2


# ---- the steps at the batch they exist for, and over the shape / option space ----------------------------------------------
def _wide_steps_match_the_oracle(case, tag, min_keep=0.75):
    """One wide critic step and one wide actor (+ temperature) step on 3xTF32, each from the case's initial state, against
    the fp32 oracle with the fp32 oracle's own distance to float64 as yardstick (tests/helpers.check_close), on the rows of
    the batch away from every ReLU kink (kink_safe / kink_safe_actor): Q values, TD target, qf_loss, actor loss, mean
    log-prob, alpha loss, log alpha, every gradient and every parameter after the Adam step. The floors are the 3xTF32
    path's stated bounds of the fixed-case tests above, in place of check_close's 1e-5: gradients 2e-5 of each tensor's
    max (TOLS: the three-product split drops the lo x lo term, ~2^-22 per product, and the weight gradients accumulate it
    over the batch), and the actor step's logged values 1e-4 (10 x TOLS, as test_wide_actor_step_matches_oracle: the actor
    loss is a batch mean of Q values, judged against its own, smaller, magnitude). The critic step's Q values, TD target
    and loss, log alpha and the parameters keep check_close's floor. min_keep: the share of the batch the kink filter
    must leave."""
    from sac_td3_cudagraphs_pytorch_b200.replay import pack_rows
    from sac_td3_cudagraphs_pytorch_b200.wide import WideActor, WideCritic
    from tests.helpers import alpha_loss_scale, check_close, check_param_after_first_adam, oracle_cuda
    gfloor, afloor = TOLS["3xtf32"][1], 10 * TOLS["3xtf32"][0]
    inp = case_inputs(case)
    full = batch_of(inp, 0, device="cuda")
    # ---- critic step
    keep = kink_safe(inp, full)
    batch = {k: v[keep] for k, v in full.items()}
    eps = inp["eps_q"][0].cuda()[keep].contiguous()
    B = int(keep.sum())
    assert B >= min_keep * inp["B"], "the kink filter should only drop a few rows"
    ag = make_agent(inp)
    o32, o64 = oracle_cuda(inp, torch.float32), oracle_cuda(inp, torch.float64)
    tq = torch.zeros(B, device="cuda")
    wc = WideCritic(ag, B, "3xtf32")
    out = wc.update_qnets(pack_rows(batch, ag.fmt), eps=eps, targ_out=tq)
    r32 = o32.update_qnets(batch, eps)
    r64 = o64.update_qnets({k: v.double() if v.is_floating_point() else v for k, v in batch.items()}, eps.double())
    torch.cuda.synchronize()
    worst = {}
    worst["TD target"] = check_close("TD target", tq, r32["_targ_q"], r64["_targ_q"])[0]
    worst["Q"] = check_close("Q", wc.q, r32["_q"].reshape(2, B), r64["_q"].reshape(2, B))[0]
    worst["qf_loss"] = check_close("qf_loss", out["loss/qf_loss"], r32["loss/qf_loss"], r64["loss/qf_loss"])[0]
    for n, p in ag.qnet_params.items():
        worst[f"critic grad {n}"] = check_close(f"grad {n}", p.grad, o32.qnet[n].grad, o64.qnet[n].grad, floor=gfloor)[0]
        check_param_after_first_adam(f"param {n}", p, o32.qnet[n], o64.qnet[n], p.grad, o32.qnet[n].grad, float(inp["hps"]["qnets_lr"]))
    dropped_q = inp["B"] - B
    # ---- actor (+ temperature) step from the same initial state
    e1, e2 = inp["eps_pi"][0][0].cuda(), inp["eps_alpha"][0][0].cuda()
    keep = kink_safe_actor(inp, full, e1)
    batch = {k: v[keep] for k, v in full.items()}
    e1, e2 = e1[keep].contiguous(), e2[keep].contiguous()
    B = int(keep.sum())
    assert B >= min_keep * inp["B"]
    ag = make_agent(inp)
    o32, o64 = oracle_cuda(inp, torch.float32), oracle_cuda(inp, torch.float64)
    wa = WideActor(ag, B, "3xtf32")
    out = wa.update_actor(pack_rows(batch, ag.fmt), eps=e1, eps_alpha=e2)
    r32 = o32.update_actor(batch, e1, e2)
    r64 = o64.update_actor({k: v.double() if v.is_floating_point() else v for k, v in batch.items()}, e1.double(), e2.double())
    torch.cuda.synchronize()
    for k in r32:
        sc = alpha_loss_scale(inp["hps"]["alpha_init"], inp["ac"]) if k == "loss/alpha_loss" else None
        worst[k] = check_close(k, out[k], r32[k], r64[k], scale=sc, floor=afloor)[0]
    for n, p in ag.actor_params.items():
        worst[f"actor grad {n}"] = check_close(f"grad {n}", p.grad, o32.actor[n].grad, o64.actor[n].grad, floor=gfloor)[0]
        check_param_after_first_adam(f"param {n}", p, o32.actor[n], o64.actor[n], p.grad, o32.actor[n].grad, float(inp["hps"]["actor_lr"]))
    if not ag.td3 and ag.autotune:
        worst["log_alpha"] = check_close("log_alpha", ag.log_alpha, o32.log_alpha, o64.log_alpha)[0]
    k = max(worst, key=worst.get)
    print(f"\n[{tag}] wide steps vs fp32 oracle: kink rows set aside {dropped_q} (critic) / {inp['B'] - B} (actor) of {inp['B']}; "
          f"worst deviation {worst[k]:.2e} ({k})")


@pytest.mark.parametrize("algo,ob,ac,B", [("sac", 11, 3, 65536), ("td3", 11, 3, 65536), ("sac", 376, 17, 16384)])
def test_wide_steps_match_the_oracle_at_config5_batch(algo, ob, ac, B):
    """BASELINE.json config 5's batch of 65 536 on Hopper shapes — every cross-CTA reduction of the wide path at full length
    (512 column-sum partials, 8 192 squared-error partials, 256 actor partials, 16 passes of the temperature gradient), both
    TMEM buffers of the tensor-core layers reused — and SAC on Humanoid shapes (376 / 17) at 16 384: heads of 34 outputs
    (the per-output loop) and a streamed first layer."""
    from tests.golden.cases import SAC, TD3
    case = dict(base=SAC if algo == "sac" else TD3, ob=ob, ac=ac, lo=[-1.0] * ac, hi=[1.0] * ac, B=B, N=B + B // 2, iters=1,
                seed=7000 + ob, over=dict(batch_size=B))
    _wide_steps_match_the_oracle(case, f"{algo} {ob}/{ac} B={B}")


def _wide_cases():
    from hypothesis import strategies as st

    from tests.golden.cases import SAC, TD3

    @st.composite
    def cases(draw):
        td3 = draw(st.booleans())
        ob, ac = draw(st.integers(1, 48)), draw(st.integers(1, 17))
        B = draw(st.sampled_from([40, 129, 300, 1000, 2047, 3000]))
        over = dict(layer_norm=draw(st.booleans()), bcq_style_targ_mix=draw(st.booleans()), batch_size=B)
        if td3:
            over.update(targ_actor_smoothing=draw(st.booleans()))
        else:
            over.update(autotune=draw(st.booleans()), alpha_init=draw(st.sampled_from([0.2, 1.0])))
        lo = [-(1.0 + 0.25 * (i % 3)) for i in range(ac)]
        hi = [0.5 + 0.5 * (i % 2) for i in range(ac)]
        case = dict(base=TD3 if td3 else SAC, ob=ob, ac=ac, lo=lo, hi=hi, B=B, N=2 * B, iters=1,
                    seed=draw(st.integers(1, 10_000)) * 11, over=over)
        return case, draw(st.sampled_from(["tc", "ffma"]))
    return cases()


def test_wide_steps_match_the_oracle_for_any_shape_and_option(monkeypatch):
    """Property test of the wide steps (3xTF32), mirroring test_gpu_property.py: O = 1..48 and A = 1..17 (first layers of
    every alignment: _first_layer takes tc_first where TMA can address the rows and wide_first elsewhere, and the draw also
    forces wide_first through B2RL_WIDE_FIRST), ragged batches up to 3 000, LayerNorm, BCQ mix, target smoothing and
    autotune on and off; the bar of check_close on the kink-safe rows (gradients: the 3xTF32 floor, see above)."""
    from hypothesis import HealthCheck, given, settings

    @settings(max_examples=25, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(drawn=_wide_cases())
    def run(drawn):
        case, first = drawn
        monkeypatch.setenv("B2RL_WIDE_FIRST", first)
        # (small batches of wide inputs: the share of rows with some unit near a kink varies more from draw to draw)
        _wide_steps_match_the_oracle(case, f"{'td3' if case['base']['prefer_td3_over_sac'] else 'sac'} {case['ob']}/{case['ac']} "
                                           f"B={case['B']} first={first} {case['over']}", min_keep=0.5)

    run()
