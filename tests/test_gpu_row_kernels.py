"""The row-group path beyond batch 256: its weight-gradient kernel (csrc/wgrad.cu, b2rl_wgrad) element by element against a
float64 restatement, and its whole critic / actor (+ temperature) steps (critic_fused / actor_fused / alpha_kernel, then
wgrad_kernel and Adam) against the fp32 and float64 oracles at batches up to 65 536.

Beyond 256 rows every cross-row-block loop of the path takes its long form: the lane-strided scalar sums of wgrad_kernel
and of alpha_kernel's last cluster run several trips per lane (nblk = ceil(B / 8) > 32), and gemm_tile restages its
32-row chunk more than once per warp (ceil(B / 8) > 32 rows per warp slice).

b2rl_wgrad is called directly through _lib on a workspace filled here (the layout of csrc/common.cuh is restated below and
its size checked against b2rl_workspace_floats). Bounds, as in test_gpu_wide_kernels.py (u = 2^-24,
gamma_k = k u / (1 - k u)):
  dW1 / dW2 / dW3   one FMA chain over the warp's ceil(B / 8) rows, then the 8 warp partials in order
                                                                       k = ceil(B/8) + 7, over sum_b |A[b][m] Bm[b][n]|
  b1 g1 be1 b2 g2 be2 b3   the nblk row-block partials in sequence     k = nblk, over sum |partials|
  qf_loss / actor loss / mean log pi   ceil(nblk / 32) partials per lane, 5 shuffle levels, / B, then the sum over the
                                       critics (running error class R);  alpha = expf(log_alpha): 2 ulp
Everything the kernel may not depend on is NaN (row columns past the net's input, dZ3 columns past the head, workspace slot
1 in an actor step, the LayerNorm partials of a net without LayerNorm, the gaps between stacked agents), every gradient
starts as NaN, and everything the step does not own must come back NaN or bitwise unchanged.

test_row_bounds_have_teeth (no GPU) shows that each bound rejects, at least tenfold, the mistakes a batch-contracting
kernel makes: a row dropped or counted twice, the neighbouring agent's rows, a partial dropped or counted twice, a mean
over 8 nblk rows instead of B.
"""
from __future__ import annotations

import ctypes as C
import math

import pytest
import torch

from tests.test_gpu_wide_kernels import (WORST, R, _fp32_within, _lib, _teeth, check, gam, guarded, r_exp, r_sum, st,
                                         untouched)

HID, MAX_OUT, RT = 256, 64, 8
# ---- the workspace layout per agent, restated from csrc/common.cuh (ws_floats, ws_carve, PART_*) ------------------------
PART_VEC = 6                            # db1 dg1 dbe1 db2 dg2 dbe2
PART_LEN = PART_VEC * HID + MAX_OUT + 8  # + db3[MAX_OUT] + {loss terms}
PART_DB3 = PART_VEC * HID
PART_SCAL = PART_VEC * HID + MAX_OUT    # [0] sum of squared errors / actor loss, [1] sum of log pi
VEC_FIELDS = ("b1", "g1", "be1", "b2", "g2", "be2")  # (the order of the PART_VEC vectors)


def nblk_of(B: int) -> int:
    return -(-B // RT)


def ws_floats(B: int) -> int:
    return 2 * B * HID * 4 + 2 * B * MAX_OUT + 2 * nblk_of(B) * PART_LEN


def ws_carve(ws: torch.Tensor, B: int, slot: int) -> dict:
    """Views of one agent's workspace: H1, H2, DZ1, DZ2 [2][B][256], DZ3 [2][B][64], PART [2][nblk][PART_LEN]."""
    bh, nb = B * HID, nblk_of(B)
    v = lambda o, *shape: ws[o:o + math.prod(shape)].view(*shape)
    tail = 8 * bh
    return dict(h1=v((0 * 2 + slot) * bh, B, HID), h2=v((1 * 2 + slot) * bh, B, HID), dz1=v((2 * 2 + slot) * bh, B, HID),
                dz2=v((3 * 2 + slot) * bh, B, HID), dz3=v(tail + slot * B * MAX_OUT, B, MAX_OUT),
                part=v(tail + 2 * B * MAX_OUT + slot * nb * PART_LEN, nb, PART_LEN))


# ---- float64 references of wgrad_kernel's outputs (plain torch; CPU or GPU) ---------------------------------------------
def gemm_ref(A, Bm, B: int) -> R:
    """C[m][n] = sum_b A[b][m] Bm[b][n] as gemm_tile sums it: k = ceil(B / 8) + 7."""
    A, Bm = A.double(), Bm.double()
    return R(A.T @ Bm, gam(nblk_of(B) + 7) * (A.abs().T @ Bm.abs()))


def vec_ref(parts) -> R:
    """Column sums of the [nblk][n] row-block partials, added in sequence."""
    return r_sum(R(parts), 0, parts.shape[0])


def mean_ref(parts, B: int) -> R:
    """(sum of the nblk scalar partials: lane-strided, then the shuffle tree) / B."""
    return r_sum(R(parts), 0, -(-parts.shape[0] // 32) + 5) / R(float(B))


# ---- b2rl_wgrad on its own ------------------------------------------------------------------------------------------------
SHAPES = {  # name: (ob, ac, td3, layer_norm)
    "hopper_sac": (11, 3, False, True),
    "hopper_td3": (11, 3, True, False),
    "humanoid_sac": (376, 17, False, True),  # critic 393 inputs: 13 m-tiles, the last partial; actor head 34 outputs
    "one_one": (1, 1, False, True),
    "in31_32": (31, 1, True, True),          # actor 31 / critic 32 inputs: one full m-tile
    "in32_33": (32, 1, False, False),        # actor 32 / critic 33: one full tile, and one tile + 1
    "a32_sac": (11, 32, False, True),        # a 64-output head: 2 full m-tiles
}
HOPPER_B = (1, 7, 8, 9, 255, 256, 257, 263, 4097, 65536, 65543)
WGRAD_CASES = (
    [(s, B, 1, 0, 0) for s in ("hopper_sac", "hopper_td3") for B in HOPPER_B]
    + [("humanoid_sac", B, 1, 0, 0) for B in (7, 257, 4097)]
    + [("one_one", B, 1, 0, 0) for B in (1, 9, 263, 4097)]
    + [("in31_32", B, 1, 0, 0) for B in (8, 257, 4097)]
    + [("in32_33", B, 1, 0, 0) for B in (9, 263, 4097)]
    + [("a32_sac", B, 1, 0, 0) for B in (255, 4097)]
    # no counter bump (bump_counter = -1); the matrices only (skip_vectors = 1)
    + [("hopper_sac", 4097, 1, 1, 0), ("hopper_td3", 257, 1, 1, 0), ("hopper_sac", 263, 1, 0, 1), ("humanoid_sac", 4097, 1, 0, 1)]
    # stacked agents, each with its own data, NaN gaps between their arena / row / workspace spans
    + [("hopper_sac", B, 3, 0, 0) for B in (1000, 4097)] + [("hopper_td3", 4097, 3, 0, 1)]
)


def _decades(g, *shape):
    """Signed values over three decades of magnitude."""
    return torch.randn(*shape, device="cuda", generator=g) * 10.0 ** (-3.0 * torch.rand(*shape, device="cuda", generator=g))


def _bits(t):
    return t.view(torch.int32).clone()


def run_wgrad(L, shape, B, n, actor_step, no_bump, skip, seed=0):
    """One b2rl_wgrad launch on hand-filled inputs; returns everything the checks need."""
    from sac_td3_cudagraphs_pytorch_b200.arena import _up4, make_layout
    lib = L.load()
    ob, ac, td3, ln = SHAPES[shape]
    lay = make_layout(ob, ac, td3, ln)
    nets = [lay.actor] if actor_step else lay.critic
    rs = _up4(2 * ob + ac + 2)
    g = torch.Generator(device="cuda").manual_seed(seed + 97 * B + 13 * n + 7 * actor_step)
    gap = 12 if n > 1 else 0  # (multiples of 4 floats)
    ars, rws = 5 * lay.region + gap, B * rs + gap
    wsf = ws_floats(B)
    assert wsf == lib.b2rl_workspace_floats(B), "the restated workspace layout disagrees with csrc/common.cuh"
    wss = wsf + gap
    ar_f, ar = guarded(n, ars)
    ar[:, :4 * lay.region] = torch.randn(n, 4 * lay.region, device="cuda", generator=g)  # regions 0-3 (region 4 stays NaN)
    rw_f, rw = guarded(n, rws)
    ws_f, ws = guarded(n, wss)
    for a in range(n):
        rows = rw[a, :B * rs].view(B, rs)
        rows[:, :nets[0].in_dim] = torch.randn(B, nets[0].in_dim, device="cuda", generator=g) * 2.0
        for k, net in enumerate(nets):
            w = ws_carve(ws[a], B, k)
            w["h1"].copy_(torch.relu(torch.randn(B, HID, device="cuda", generator=g)))
            w["h2"].copy_(torch.relu(torch.randn(B, HID, device="cuda", generator=g)))
            w["dz1"].copy_(_decades(g, B, HID))
            w["dz2"].copy_(_decades(g, B, HID))
            w["dz3"][:, :net.out_dim] = _decades(g, B, net.out_dim)
            p = w["part"]
            for v in (range(PART_VEC) if ln else (0, 3)):
                p[:, v * HID:(v + 1) * HID] = _decades(g, nblk_of(B), HID)
            p[:, PART_DB3:PART_DB3 + net.out_dim] = _decades(g, nblk_of(B), net.out_dim)
            if actor_step:
                p[:, PART_SCAL] = torch.randn(nblk_of(B), device="cuda", generator=g) * 3.0
                p[:, PART_SCAL + 1] = torch.randn(nblk_of(B), device="cuda", generator=g) * 4.0 - 2.0
            else:  # (a sum of squared TD errors; the log-pi field is not the critic step's)
                p[:, PART_SCAL] = torch.rand(nblk_of(B), device="cuda", generator=g) * 5.0
    la_f, la = guarded(n, 5)
    la[:, 0] = torch.tensor([-1.3, 0.4, -0.2][:n], device="cuda")
    o_f, out = guarded(n, 8)
    ctr = (torch.arange(n * 8, device="cuda", dtype=torch.int64).view(n, 8) * 3 + 5)
    ctr[:, L.CTR_TICKET] = 0
    lo, hi = -torch.ones(ac, device="cuda"), torch.ones(ac, device="cuda")
    bump = -1 if no_bump else (L.CTR_PI if actor_step else L.CTR_Q)
    before = dict(ar=_bits(ar[:, :4 * lay.region]), rw=_bits(rw_f), ws=_bits(ws_f), ctr=ctr.clone())
    a = L.UpdateArgs()
    a.hp = L.Hyper(td3=int(td3), gamma=0.99, targ_ent=-float(ac), seed=1)
    a.fmt = L.RowFmt(ob, ac, rs, 0)
    a.actor = lay.actor.c_struct()
    a.critic[0], a.critic[1] = lay.critic[0].c_struct(), lay.critic[1].c_struct()
    a.batch, a.n_agents, a.agent_base = B, n, 0
    a.region_stride, a.arena_agent_stride = lay.region, ars
    a.arena, a.rows, a.rows_agent_stride = ar.data_ptr(), rw.data_ptr(), rws
    a.min_ac, a.max_ac, a.log_alpha, a.counters = lo.data_ptr(), hi.data_ptr(), la.data_ptr(), ctr.data_ptr()
    a.workspace, a.workspace_agent_stride, a.out = ws.data_ptr(), wss, out.data_ptr()
    L.check(lib.b2rl_wgrad(C.byref(a), int(actor_step), bump, int(skip), st()), "wgrad")
    torch.cuda.synchronize()
    return dict(lay=lay, nets=nets, rs=rs, ar_f=ar_f, ar=ar, rw_f=rw_f, rw=rw, ws=ws, ws_f=ws_f, la=la, o_f=o_f, out=out, ctr=ctr,
                bump=bump, before=before, td3=td3)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,B,n,no_bump,skip", WGRAD_CASES)
@pytest.mark.parametrize("actor_step", [0, 1])
def test_wgrad_matches_float64(shape, B, n, no_bump, skip, actor_step):
    """b2rl_wgrad, critic step (both critics, workspace slots 0 and 1) or actor step (slot 0; slot 1 NaN): every gradient
    element the step owns within its float64 bound, the w2n shadow bitwise the transpose of w2t, the scalar outputs, and
    nothing else written — the other nets' spans, the padding between tensors, regions 0-3, the inputs, the other out
    fields, the other counter slots."""
    L = _lib()
    r = run_wgrad(L, shape, B, n, actor_step, no_bump, skip)
    lay, nets, rs, ar, ws, out = r["lay"], r["nets"], r["rs"], r["ar"], r["ws"], r["out"]
    G4 = 4 * lay.region
    owned = torch.zeros_like(ar, dtype=torch.bool)
    o_own = torch.zeros_like(out, dtype=torch.bool)
    for a in range(n):
        tag = f"{shape} {'actor' if actor_step else 'critic'} B={B} n={n} agent {a}"
        G = ar[a, G4:G4 + lay.region]
        x0 = r["rw"][a, :B * rs].view(B, rs)
        for k, net in enumerate(nets):
            w = ws_carve(ws[a], B, k)
            gv = lambda f, *shape: G[net.off[f]:net.off[f] + net.numel(f)].view(*shape)
            own = lambda f: owned[a, G4 + net.off[f]:G4 + net.off[f] + net.numel(f)].fill_(True)
            t = f"{tag} net {k}"
            check("wgrad dW1", t, gv("w1t", net.in_dim, HID), gemm_ref(x0[:, :net.in_dim], w["dz1"], B))
            check("wgrad dW2", t, gv("w2t", HID, HID), gemm_ref(w["h1"], w["dz2"], B))
            check("wgrad dW3", t, gv("w3", net.out_dim, HID), gemm_ref(w["dz3"][:, :net.out_dim], w["h2"], B))
            assert torch.equal(gv("w2n", HID, HID).view(torch.int32), gv("w2t", HID, HID).t().contiguous().view(torch.int32)), \
                t + ": the w2n shadow is not bitwise the transpose of w2t"
            for f in ("w1t", "w2t", "w3", "w2n"):
                own(f)
            if skip:
                continue
            for v, f in enumerate(VEC_FIELDS):
                if net.off[f] >= 0:
                    check("wgrad b/g/be", f"{t} d{f}", gv(f, HID), vec_ref(w["part"][:, v * HID:(v + 1) * HID]))
                    own(f)
            check("wgrad b3", t, gv("b3", net.out_dim), vec_ref(w["part"][:, PART_DB3:PART_DB3 + net.out_dim]))
            own("b3")
        if skip:
            continue
        p0 = ws_carve(ws[a], B, 0)["part"]
        if actor_step:
            check("wgrad scalars", tag + " actor loss", out[a, L.OUT_ACTOR_LOSS], mean_ref(p0[:, PART_SCAL], B))
            check("wgrad scalars", tag + " mean log pi", out[a, L.OUT_LOGPI_MEAN], mean_ref(p0[:, PART_SCAL + 1], B))
            o_own[a, [L.OUT_ACTOR_LOSS, L.OUT_LOGPI_MEAN]] = True
            if not r["td3"]:
                check("wgrad scalars", tag + " alpha", out[a, L.OUT_ALPHA], r_exp(R(r["la"][a, 0])))
                o_own[a, L.OUT_ALPHA] = True
        else:
            p1 = ws_carve(ws[a], B, 1)["part"]
            check("wgrad scalars", tag + " qf_loss", out[a, L.OUT_QF_LOSS], mean_ref(p0[:, PART_SCAL], B) + mean_ref(p1[:, PART_SCAL], B))
            o_own[a, L.OUT_QF_LOSS] = True
    # nothing else was written: region 4 outside the step's own tensors (padding, the other nets), the agent gaps, the
    # guard bands; regions 0-3 and the inputs bitwise; the out fields the step does not own
    notg = ~owned
    notg[:, :G4] = False
    untouched(r["ar_f"], ar, notg, "arena region 4 / agent gaps")
    assert torch.equal(_bits(ar[:, :G4]), r["before"]["ar"]), "arena regions 0-3 changed"
    assert torch.equal(_bits(r["rw_f"]), r["before"]["rw"]) and torch.equal(_bits(r["ws_f"]), r["before"]["ws"]), "an input changed"
    untouched(r["o_f"], out, ~o_own, "out")
    want = r["before"]["ctr"].clone()
    if r["bump"] >= 0:
        want[:, r["bump"]] += 1
    assert torch.equal(r["ctr"], want), f"counters {r['ctr'].tolist()} != {want.tolist()}"


# ---- the row-group steps beyond 256 against the oracles ----------------------------------------------------------------------
def _row_steps_match_the_oracle(case, tag, min_keep=0.75):
    """One row-path critic step and one actor (+ temperature) step through the Agent API with injected noise, each from
    the case's initial state, against the fp32 oracle with the fp32 oracle's own distance to float64 as yardstick
    (tests/helpers.check_close, its default bar: floor 1e-5, factor 4), on the rows away from every ReLU kink (kink_safe /
    kink_safe_actor): Q values, TD target, qf_loss, the logged actor values (alpha_loss judged against alpha * A,
    helpers.alpha_loss_scale), log alpha, every gradient and every parameter after the first Adam step. A clipped actor
    gradient is not compared (the oracle's .grad holds the clipped gradient, the arena the unclipped one): its logged
    values are."""
    from tests.golden.cases import case_inputs
    from tests.helpers import (alpha_loss_scale, batch_of, check_close, check_param_after_first_adam, kink_safe, kink_safe_actor,
                               make_agent, oracle_cuda)
    inp = case_inputs(case)
    full = batch_of(inp, 0, device="cuda")
    f64 = lambda d: {k: v.double() if v.is_floating_point() else v for k, v in d.items()}
    worst = {}

    def note(what, d):
        worst[what] = d[:2]
    # ---- critic step
    keep = kink_safe(inp, full)
    batch = {k: v[keep] for k, v in full.items()}
    eps = inp["eps_q"][0].cuda()[keep].contiguous()
    B = int(keep.sum())
    assert B >= min_keep * inp["B"], "the kink filter should only drop a few rows"
    ag = make_agent(inp)
    o32, o64 = oracle_cuda(inp, torch.float32), oracle_cuda(inp, torch.float64)
    tq, qv = torch.zeros(B, device="cuda"), torch.zeros(2, B, device="cuda")
    out = ag.update_qnets(batch, eps=eps, dbg_targ_q=tq, dbg_q=qv)
    r32 = o32.update_qnets(batch, eps)
    r64 = o64.update_qnets(f64(batch), eps.double())
    torch.cuda.synchronize()
    note("TD target", check_close("TD target", tq, r32["_targ_q"], r64["_targ_q"]))
    note("Q", check_close("Q", qv, r32["_q"].reshape(2, B), r64["_q"].reshape(2, B)))
    note("qf_loss", check_close("qf_loss", out["loss/qf_loss"], r32["loss/qf_loss"], r64["loss/qf_loss"]))
    for n, p in ag.qnet_params.items():
        note(f"critic grad {n}", check_close(f"grad {n}", p.grad, o32.qnet[n].grad, o64.qnet[n].grad))
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
    out = ag.update_actor(batch, eps=e1, eps_alpha=e2)
    r32 = o32.update_actor(batch, e1, e2)
    r64 = o64.update_actor(f64(batch), e1.double(), e2.double())
    torch.cuda.synchronize()
    for k in r32:
        sc = alpha_loss_scale(inp["hps"]["alpha_init"], inp["ac"]) if k == "loss/alpha_loss" else None
        note(k, check_close(k, out[k], r32[k], r64[k], scale=sc))
    if not inp["hps"]["clip_norm"] > 0:
        for n, p in ag.actor_params.items():
            note(f"actor grad {n}", check_close(f"grad {n}", p.grad, o32.actor[n].grad, o64.actor[n].grad))
            check_param_after_first_adam(f"param {n}", p, o32.actor[n], o64.actor[n], p.grad, o32.actor[n].grad,
                                         float(inp["hps"]["actor_lr"]))
    if not ag.td3 and ag.autotune:
        note("log_alpha", check_close("log_alpha", ag.log_alpha, o32.log_alpha, o64.log_alpha))
    k32 = max(worst, key=lambda k: worst[k][0])
    k64 = max(worst, key=lambda k: worst[k][1])
    print(f"\n[{tag}] row steps: kink rows set aside {dropped_q} (critic) / {inp['B'] - B} (actor) of {inp['B']}; worst deviation "
          f"from the fp32 oracle {worst[k32][0]:.2e} ({k32}), from float64 {worst[k64][1]:.2e} ({k64})")


@pytest.mark.gpu
@pytest.mark.parametrize("algo,ob,ac,B", [("sac", 11, 3, 65536), ("td3", 11, 3, 65536), ("sac", 376, 17, 16384)])
def test_row_steps_match_the_oracle_at_config5_batch(algo, ob, ac, B):
    """BASELINE.json config 5's batch of 65 536 on Hopper shapes (nblk = 8 192 row blocks: 256 lane-strided trips in the
    scalar sums of wgrad_kernel and alpha_kernel, 32 chunks per gemm_tile warp slice), and SAC on Humanoid shapes (376 /
    17) at 16 384: the streamed-first-layer instantiation of critic_fused / actor_fused / alpha_kernel and a 34-output
    head."""
    from tests.golden.cases import SAC, TD3
    case = dict(base=SAC if algo == "sac" else TD3, ob=ob, ac=ac, lo=[-1.0] * ac, hi=[1.0] * ac, B=B, N=B + B // 2, iters=1,
                seed=7100 + ob, over=dict(batch_size=B))
    _row_steps_match_the_oracle(case, f"{algo} {ob}/{ac} B={B}")


def _row_cases():
    from hypothesis import strategies as st

    from tests.golden.cases import SAC, TD3

    @st.composite
    def cases(draw):
        td3 = draw(st.booleans())
        ob, ac = draw(st.integers(1, 48)), draw(st.integers(1, 17))
        B = draw(st.sampled_from([257, 300, 1000, 2047, 3000, 4097]))
        over = dict(layer_norm=draw(st.booleans()), bcq_style_targ_mix=draw(st.booleans()),
                    clip_norm=draw(st.sampled_from([0.0, 0.0, 0.25])), batch_size=B)
        if td3:
            over.update(targ_actor_smoothing=draw(st.booleans()))
        else:
            over.update(autotune=draw(st.booleans()), alpha_init=draw(st.sampled_from([0.2, 1.0])))
        lo = [-(1.0 + 0.25 * (i % 3)) for i in range(ac)]
        hi = [0.5 + 0.5 * (i % 2) for i in range(ac)]
        return dict(base=TD3 if td3 else SAC, ob=ob, ac=ac, lo=lo, hi=hi, B=B, N=2 * B, iters=1,
                    seed=draw(st.integers(1, 10_000)) * 13, over=over)
    return cases()


@pytest.mark.gpu
def test_row_steps_match_the_oracle_for_any_shape_and_option():
    """Property test of the row steps beyond 256, mirroring test_gpu_property.py: O = 1..48, A = 1..17 (first layers staged
    in shared memory and streamed), ragged batches from 257 to 4 097, LayerNorm, BCQ mix, target smoothing, autotune and
    gradient clipping on and off; check_close's bar on the kink-safe rows."""
    from hypothesis import HealthCheck, given, settings

    @settings(max_examples=25, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(case=_row_cases())
    def run(case):
        # (small inputs: the share of rows with some unit near a kink varies more from draw to draw)
        _row_steps_match_the_oracle(case, f"{'td3' if case['base']['prefer_td3_over_sac'] else 'sac'} {case['ob']}/{case['ac']} "
                                          f"B={case['B']} {case['over']}", min_keep=0.5)

    run()


@pytest.mark.gpu
def test_report_worst_wgrad_ratios():
    """(runs after the b2rl_wgrad tests of this module) the worst deviation / bound ratio of each output kind."""
    for k, v in sorted(WORST.items()):
        if k.startswith("wgrad"):
            print(f"worst dev/bound {k:16s} {v:.3f}")


# ---- the bounds have teeth (no GPU) --------------------------------------------------------------------------------------
def test_row_bounds_have_teeth():
    """At small shapes on the CPU: each bound accepts an fp32 evaluation in another summation order and rejects, at least
    tenfold, a row dropped (the last of a warp slice, the last of the batch), the last valid row counted twice (stage_tile
    pads a ragged row block by repeating it), the neighbouring agent's rows, a row-block partial dropped or counted twice,
    and a mean over 8 nblk rows instead of B."""
    g = torch.Generator().manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g)
    dec = lambda *s: rn(*s) * 10.0 ** (-3.0 * torch.rand(*s, generator=g))
    # weight gradients: B = 100 rows, warp slices of 13
    B, M = 100, 40
    bs = nblk_of(B)
    X = [torch.relu(rn(B, M)) for _ in range(2)]
    D = [dec(B, HID) for _ in range(2)]
    ref = gemm_ref(X[0], D[0], B)
    perm = torch.randperm(B, generator=g)
    _fp32_within("dW, fp32 in another order", X[0][perm].T @ D[0][perm], ref)
    x, d = X[0].double(), D[0].double()
    for name, rows in (("last row of warp slice 0", bs - 1), ("last row of the batch", B - 1)):
        k = torch.ones(B, dtype=torch.bool)
        k[rows] = False
        _teeth(f"dW, {name} dropped", x[k].T @ d[k], ref)
    _teeth("dW, last valid row counted twice", x.T @ d + torch.outer(x[-1], d[-1]), ref)
    _teeth("dW, neighbouring agent's rows", X[1].double().T @ D[1].double(), ref)
    _teeth("dW, neighbouring agent's A rows", X[1].double().T @ d, ref)
    # column vectors: 65 row-block partials
    part = dec(65, HID)
    ref = vec_ref(part)
    _fp32_within("vector, fp32 in another order", part.flip(0).sum(0), ref)
    _teeth("vector, partial dropped", part[1:].double().sum(0), ref)
    _teeth("vector, partial counted twice", part.double().sum(0) + part[40].double(), ref)
    # scalars at B = 4 097 (nblk = 513: 17 trips per lane)
    B = 4097
    nb = nblk_of(B)
    p0, p1 = torch.rand(nb, generator=g) * 5, torch.rand(nb, generator=g) * 5
    ref = mean_ref(p0, B) + mean_ref(p1, B)
    _fp32_within("qf_loss, fp32 in another order", p0.flip(0).sum() / B + p1.sum() / B, ref)
    _teeth("qf_loss, mean over 8 nblk rows", (p0.double().sum() + p1.double().sum()) / (RT * nb), ref)
    _teeth("qf_loss, partial dropped", (p0[1:].double().sum() + p1.double().sum()) / B, ref)
    _teeth("qf_loss, partial counted twice", (p0.double().sum() + p0[500].double() + p1.double().sum()) / B, ref)
    lp = rn(nb) * 4 - 2
    ref = mean_ref(lp, B)
    _teeth("mean log pi, mean over 8 nblk rows", lp.double().sum() / (RT * nb), ref)
