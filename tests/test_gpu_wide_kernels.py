"""Every entry point of the wide path's own kernels (csrc/wide.cu, and the critic head fused into tc_linear.cu) against a
float64 restatement, element by element, at the sizes where their indexing and reductions change.

The kernels are called directly through _lib with fp32 inputs; the reference is computed in float64 from those same fp32
values. Each output gets its own bound (u = 2^-24, the unit roundoff of fp32; gamma_k = k u / (1 - k u)):

  - Sums: |got - ref| <= gamma_k * sum|terms|, k the longest chain of fp32 roundings any term passes through in the
    kernel's loop structure. sum|terms| rather than max|ref|, so that cancellation can neither hide nor fake a failure.
      head dot products (wide_policy_head, wide_q_head)   8 FMAs per lane + 5 shuffle levels + the bias        k = 14
      wide_dqda                                           8 FMAs per lane + 5 shuffle levels                   k = 13
      tc_linear_q's fused head                            up to 256 FMAs along the row (two halves) + 1 + bias k = 258
      sq_part (8 rows per partial)                        8 rows in sequence (wide_q_head) / 3 levels (tc)     k = 7
      wide_actor_loss / wide_actor_head_bwd partials      5 shuffle levels + 8 warps in sequence               k = 12
      wide_colsum                                         ceil(P / S) loads per slice, then S slices; S = 32 for P >= 64
                                                          (1 024 threads), else 8                              k = ceil(P/S) + S - 1
      wide_critic_scalars                                 2 ceil(P / 256) per thread, then min(P, 256) in sequence, / M
                                                                                                               k = 2 ceil(P/256) + min(P, 256)
      wide_actor_scalars                                  P partials in sequence, / M                          k = P
      wide_alpha_grad                                     one rounding per term (-logpi - targ_ent), ceil(M / 256) per
                                                          thread, then min(M, 256) in sequence                 k = ceil(M/256) + min(M, 256)
    A product of a sum with a scalar, or a sum of rounded terms, adds the terms' own bounds first (running error
    analysis, class R of tests/helpers.py: every fp32 operation rounds once, |d fl(x)| <= u |x|; an FMA rounds less, so the bound
    holds whether or not the compiler contracts).
  - Transcendentals (policy.cuh: tanhf, expf, logf): the CUDA C++ Programming Guide's maximum ulp errors of the
    single-precision functions — tanhf 2, expf 2, logf 1 — with 1 ulp <= 2u |result|, plus the input's bound times the
    derivative. This is tighter than the behaviour-policy tests' rtol 1e-5 / atol 2e-6 away from saturation and follows
    the fp32 cancellation where there is one.
  - Saturated samples: where tanh(x) is within 1e-3 of +-1, fp32 1 - y^2 cancels and log pi moves legitimately by up
    to ~ 2 |dy| scale / (scale (1 - y^2) + 1e-6) (|dy| ~ 4u from tanhf's 2 ulp). The running bound carries exactly that
    term; such samples are counted and their worst ratio is reported separately.
  - tc_linear_q's hidden layer: the 3xTF32 product's stated bound of test_gpu_tc.py (4e-6 of the layer's largest
    output), propagated through w3.

Every output buffer lies inside a NaN guard band of GUARD floats and starts as NaN: each element a kernel owns must come
back finite, and every element it does not own — the guard band, the columns past a head's outputs, the save slots TD3
does not use, the LayerNorm offsets of a job without LayerNorm, the log fields and gradient entries a scalar kernel must
not touch — must still be NaN. The worst deviation / bound ratio of each kernel is printed.

test_bounds_have_teeth (no GPU) shows that each bound rejects, at least tenfold, plausible mistakes applied to the same
float64 references: a partial dropped or counted twice, the neighbouring agent's parameters or rows, 2/M taken over all
agents' rows, the tie gradient sent to critic 1, another agent's target entropy.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests.helpers import FLOOR, GUARD, WIDEN, R, U, gam, guarded, r_sum, untouched  # noqa: F401

ULP_TANH, ULP_EXP, ULP_LOG = 2, 2, 1  # CUDA C++ Programming Guide, single-precision mathematical functions
MAX_OUT, HID = 64, 256
LOG_STD_MIN, LOG_STD_MAX = -5.0, 2.0
f32 = lambda x: float(np.float32(x))
LOG_SQRT_2PI = f32(0.9189385332046727)
SAT = 1e-3  # |1 - y^2| below this: a saturated sample


# ---- running error analysis (gam, R, r_sum: tests/helpers.py) ---------------------------------------------------------
def r_tanh(a: R) -> R:
    v = torch.tanh(a.v)
    return R(v, (1 - v * v) * a.e + 2 * ULP_TANH * U * v.abs())


def r_exp(a: R) -> R:
    v = torch.exp(a.v)
    return R(v, v * torch.expm1(a.e) + 2 * ULP_EXP * U * v * torch.exp(a.e))


def r_log(a: R) -> R:
    v = torch.log(a.v)
    return R(v, -torch.log1p(-a.e / a.v) + 2 * ULP_LOG * U * v.abs())


def r_clamp(a: R, lo, hi) -> R:  # (1-Lipschitz, exact in fp32)
    if not torch.is_tensor(lo):
        return R(a.v.clamp(lo, hi), a.e)
    return R(torch.minimum(torch.maximum(a.v, lo), hi), a.e)


def r_dot(x, w, b, k):
    """x [M][K] . w [O][K]^T + b [O]: a sum whose longest chain is k roundings."""
    x, w, b = x.double(), w.double(), b.double()
    return R(x @ w.T + b, gam(k) * (x.abs() @ w.abs().T + b.abs()))


def group_sum(a: R, g: int, k: int) -> R:
    """Sums over consecutive groups of g rows (a ragged last group is padded with exact zeros)."""
    n = a.v.shape[0]
    pad = (-n) % g
    v = torch.cat([a.v, a.v.new_zeros(pad, *a.v.shape[1:])]).view(-1, g, *a.v.shape[1:])
    e = torch.cat([a.e, a.e.new_zeros(pad, *a.e.shape[1:])]).view(-1, g, *a.e.shape[1:])
    return r_sum(R(v, e), 1, k)


# ---- float64 references (plain torch functions of the kernels' fp32 inputs; CPU or GPU) --------------------------------
def policy_head_ref(h2, w3, b3, eps, lo, hi, A, td3, smoothing=False, std=0.0, c=0.0, u=None):
    """wide_policy_head for one agent: head u = h2 . w3^T + b3, then TD3's tanh action (+ clipped, clamped smoothing
    noise) or SAC's tanh-Gaussian sample and log-prob (policy.cuh, in its operation order). Returns R-valued
    {act, logp, eps, sigma, y, th} (SAC) / {act, th} (TD3). u: the head's output as an R, when it is computed elsewhere
    (an h2 that carries its own bound)."""
    u = r_dot(h2, w3, b3, 14) if u is None else u
    lo, hi = lo.double(), hi.double()
    scale, bias = (R(hi) - R(lo)) * 0.5, (R(hi) + R(lo)) * 0.5
    if td3:
        th = r_tanh(u[:, :A])
        act = th * scale + bias
        if smoothing:
            n = r_clamp(R(eps) * f32(std), -f32(c), f32(c))
            act = r_clamp(act + n, lo, hi)
        return dict(act=act, th=th)
    mu, raw = u[:, :A], u[:, A:2 * A]
    th = r_tanh(raw)
    ls = LOG_STD_MIN + (0.5 * (LOG_STD_MAX - LOG_STD_MIN)) * (th + 1.0)
    sigma = r_exp(ls)
    es = R(eps) * sigma
    x = mu + es
    y = r_tanh(x)
    act = y * scale + bias
    d = R(es.v, es.e + U * x.v.abs() + U * es.v.abs())  # fl(x - mu): eps * sigma, x's rounding and one more
    logn = -((d * d) / (2.0 * (sigma * sigma))) - r_log(sigma) - LOG_SQRT_2PI
    corr = r_log(scale * (1.0 - y * y) + f32(1e-6))
    lp = logn - corr
    return dict(act=act, logp=r_sum(lp, 1, max(A - 1, 1)), eps=R(eps), sigma=sigma, y=y, th=th, sat=(1 - y.v * y.v).abs() < SAT)


def q_target_ref(q: R, qn0, qn1, logp, log_alpha, r, d, gamma, M, td3, bcq):
    """The critic head's online mode (agents/agent.py:212-233): TD target y, dLoss/dQ = 2 (q - y) / M, (q - y)^2.
    qn0, qn1, logp: fp32 inputs, or R values that carry their own bounds (min / max move by at most the larger one)."""
    qn0, qn1 = R.of(qn0), R.of(qn1)
    e = torch.maximum(qn0.e, qn1.e)
    qmin, qmax = R(torch.minimum(qn0.v, qn1.v), e), R(torch.maximum(qn0.v, qn1.v), e)
    qp = 0.75 * qmin + 0.25 * qmax if bcq else qmin
    if not td3:
        qp = qp - r_exp(R(log_alpha)) * R.of(logp)
    y = R(r) + ((1.0 - R(d)) * f32(gamma)) * qp
    dlt = q - y
    return dict(y=y, dz=dlt * (R(2.0) / R(float(M))), sq=dlt * dlt)


def colsum_ref(part, k):
    """part [P][3][256] -> the three column sums [3][256]."""
    return r_sum(R(part), 0, k)


def colsum_k(P):
    s = 32 if P >= 64 else 8
    return math.ceil(P / s) + s - 1


def critic_scalars_ref(sq0, sq1, M):
    """sq0 / sq1 [P][2] -> (qf_loss, d b3_0, d b3_1)."""
    P = sq0.shape[0]
    k = 2 * math.ceil(P / 256) + min(P, 256)
    loss = r_sum(R(sq0[:, 0].double() + sq1[:, 0].double(), gam(1) * (sq0[:, 0].double() + sq1[:, 0].double()).abs()), 0, k)
    return loss / R(float(M)), r_sum(R(sq0[:, 1]), 0, k), r_sum(R(sq1[:, 1]), 0, k)


def actor_loss_ref(q0, q1, logp, log_alpha, td3, M):
    """Per row: loss term and dLoss/dQ_k (the whole gradient to critic 0 on ties, as torch.min); per 256-row CTA: sums."""
    q0 = q0.double()
    inv, e_inv = 1.0 / M, U / M  # fl(1 / M)
    if td3:
        return dict(d0=R(torch.full_like(q0, -inv), torch.full_like(q0, e_inv)), d1=None, loss=R(-q0), lp=R(torch.zeros_like(q0)))
    q1 = q1.double()
    first = q0 <= q1
    d0 = R(torch.where(first, -inv, 0.0), torch.where(first, e_inv, 0.0))
    d1 = R(torch.where(first, 0.0, -inv), torch.where(first, 0.0, e_inv))
    loss = r_exp(R(log_alpha)) * R(logp) - R(torch.where(first, q0, q1))
    return dict(d0=d0, d1=d1, loss=loss, lp=R(logp))


def head_bwd_ref(dqda0, dqda1, save, lo, hi, log_alpha, td3, A, M, recip=False):
    """wide_actor_head_bwd for one agent: du [M][out] from dQ/da and the saved sampling intermediates (policy.cuh
    gauss_backward in its operation order). dQ/da and save may be R values: save then is the sequence (eps, sigma, y, th).
    recip: c_pi = alpha * fl(1 / M), the fused actor's rounding, instead of alpha / M."""
    ga = R.of(dqda0) if dqda1 is None else R.of(dqda0) + R.of(dqda1)
    scale = (R(hi.double()) - R(lo.double())) * 0.5
    sv = save if isinstance(save, (list, tuple)) else [save[:, i] for i in range(4)]
    th = R.of(sv[3])
    if td3:
        return dict(du=ga * scale * (1.0 - th * th), sat=torch.zeros_like(ga.v, dtype=torch.bool))
    eps, sigma, y = R.of(sv[0]), R.of(sv[1]), R.of(sv[2])
    c_pi = r_exp(R(log_alpha)) * (R(1.0) / R(float(M))) if recip else r_exp(R(log_alpha)) / R(float(M))
    omy = 1.0 - y * y
    dcorr = (-2.0 * y * scale) / (scale * omy + f32(1e-6))
    gx = (ga * scale - c_pi * dcorr) * omy
    g_raw = ((gx * eps - c_pi / sigma) * sigma) * (0.5 * (LOG_STD_MAX - LOG_STD_MIN)) * (1.0 - th * th)
    return dict(du=R(torch.cat([gx.v, g_raw.v], 1), torch.cat([gx.e, g_raw.e], 1)),
                sat=torch.cat([omy.v.abs() < SAT] * 2, 1))


def alpha_grad_ref(logp2, log_alpha, targ_ent):
    M = logp2.shape[0]
    t = -logp2.double() - f32(targ_ent)
    s = r_sum(R(t, U * t.abs()), 0, math.ceil(M / 256) + min(M, 256))
    return r_exp(R(log_alpha)) * (s / R(float(M)))


# ---- device helpers -----------------------------------------------------------------------------------------------------
WORST: dict = {}


def check(kernel, what, got, ref: R, sat=None):
    """|got - ref.v| <= ref.e (widened) element-wise; saturated samples (mask) reported on their own."""
    got = got.detach()
    assert torch.isfinite(got).all(), f"{kernel} {what}: an owned element was not written (or is not finite)"
    dev = (got.double() - ref.v).abs()
    ratio = dev / (WIDEN * ref.e + FLOOR)
    if sat is None:
        sat = torch.zeros_like(ratio, dtype=torch.bool)
    r_ok = float(ratio[~sat].max()) if bool((~sat).any()) else 0.0
    r_sat = float(ratio[sat].max()) if bool(sat.any()) else 0.0
    WORST[kernel] = max(WORST.get(kernel, 0.0), r_ok, r_sat)
    msg = f"{kernel} {what}: worst dev/bound {r_ok:.3f}"
    if bool(sat.any()):
        msg += f"; {int(sat.sum())} saturated samples, worst {r_sat:.3f}"
    print(msg)
    assert r_ok <= 1.0 and r_sat <= 1.0, msg


def _lib():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    L.load()
    L.init_device(torch.device("cuda"))
    return L


def hp_table(algo, n, gamma=None, td3_std=None, td3_c=None, targ_ent=None, A=3):
    """b2rl_agent_hp_t rows (population.agent_hp_values / agent_hp_table) with per-agent values."""
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.population import agent_hp_table, agent_hp_values
    hps = (td3_hps if algo == "td3" else sac_hps)(batch_size=256)
    over = {k: v for k, v in dict(gamma=gamma, td3_std=td3_std, td3_c=td3_c, targ_ent=targ_ent).items() if v is not None}
    vals = agent_hp_values(hps, n, A, over)
    return torch.from_numpy(agent_hp_table(vals, algo == "td3")).cuda(), vals


def stack(L, n, base, ps=0, alpha=0, ctr=0, out=0, hp=None, lo=0):
    return L.Stack(n, base, ps, lo, alpha, ctr, out, None if hp is None else hp.data_ptr())


def st():
    return torch.cuda.current_stream().cuda_stream


# ---- wide_policy_head -----------------------------------------------------------------------------------------------------
POLICY_CASES = (
    [("sac", A, 0, 1, 257, False) for A in (1, 3, 4, 5, 17, 32)]
    + [("td3", A, s, 1, 257, False) for A in (1, 3, 4, 5, 17, 32) for s in (0, 1)]
    + [("sac", 3, 0, 1, M, False) for M in (1, 63, 64, 65)]
    + [("td3", 4, 1, 1, M, False) for M in (7, 64, 4097)]
    + [("sac", 17, 0, 3, 200, True), ("sac", 4, 0, 3, 200, True), ("td3", 5, 1, 3, 200, True), ("td3", 3, 1, 3, 200, False),
       ("td3", 32, 1, 3, 129, True)]
)


def run_policy_head(L, algo, A, smoothing, n, M, table, seed=0, src_off=None):
    """One wide_policy_head launch on random inputs (heads that saturate, asymmetric bounds); returns inputs and outputs."""
    g = torch.Generator(device="cuda").manual_seed(1000 * A + 10 * n + M + seed)
    td3 = algo == "td3"
    out_dim = A if td3 else 2 * A
    O = 11
    rs = (2 * O + A + 2 + 3) & ~3
    src = O + A + 2 if src_off is None else src_off
    ldn = O + A + 3  # (three padding columns the kernel must leave alone)
    ps = out_dim * HID + 68
    P = torch.randn(n, ps, device="cuda", generator=g) / 8.0
    P[:, out_dim * HID:out_dim * HID + out_dim] = 0.3 * torch.randn(n, out_dim, device="cuda", generator=g)
    h2 = torch.relu(torch.randn(n * M, HID, device="cuda", generator=g))
    rows = torch.randn(n * M, rs, device="cuda", generator=g)
    lo = -0.5 - torch.rand(A, device="cuda", generator=g)
    hi = 0.2 + 1.5 * torch.rand(A, device="cuda", generator=g)
    eps = torch.randn(n * M, A, device="cuda", generator=g)
    ctr = torch.zeros(n, 8, dtype=torch.int64, device="cuda")
    xn_f, xn = guarded(n * M, ldn)
    lp_f, lp = guarded(n * M)
    sv_f, sv = guarded(n * M, 4, A)
    eo_f, eo = guarded(n * M, A)
    p = L.WidePolicy()
    p.h2, p.w3, p.b3 = h2.data_ptr(), P.data_ptr(), P.data_ptr() + 4 * out_dim * HID
    p.rows, p.min_ac, p.max_ac = rows.data_ptr(), lo.data_ptr(), hi.data_ptr()
    p.eps, p.eps_out, p.xn, p.logp, p.save = eps.data_ptr(), eo.data_ptr(), xn.data_ptr(), None if td3 else lp.data_ptr(), sv.data_ptr()
    p.counters = ctr.data_ptr()
    p.M, p.O, p.A, p.out_dim, p.row_stride, p.ldn, p.src_off = M, O, A, out_dim, rs, ldn, src
    p.td3, p.smoothing, p.counter_idx, p.stream_id = int(td3), smoothing, L.CTR_Q, 1
    p.td3_std, p.td3_c, p.seed, p.agent = 0.2, 0.5, 1234, 7
    hp, vals = None, None
    if table:
        sweep = dict(td3_std=[0.3, 0.6, 0.1][:n], td3_c=[0.5, 0.25, 0.05][:n]) if td3 else dict(gamma=[0.9, 0.8, 0.7][:n])
        hp, vals = hp_table(algo, n, A=A, **sweep)
    stk = stack(L, n, 7, ps=ps, ctr=8, hp=hp) if n > 1 or table else None
    L.check(L.load().b2rl_wide_policy_head(C.byref(p), None if stk is None else C.byref(stk), st()), "wide_policy_head")
    torch.cuda.synchronize()
    stds = [f32(v["td3_std"]) for v in vals] if (table and td3) else [f32(0.2)] * n
    cs = [f32(v["td3_c"]) for v in vals] if (table and td3) else [f32(0.5)] * n
    return dict(P=P, h2=h2, rows=rows, lo=lo, hi=hi, eps=eps, xn=xn, xn_f=xn_f, lp=lp, lp_f=lp_f, sv=sv, sv_f=sv_f, eo=eo, eo_f=eo_f,
                O=O, src=src, ldn=ldn, out_dim=out_dim, stds=stds, cs=cs)


@pytest.mark.gpu
@pytest.mark.parametrize("algo,A,smoothing,n,M,table", POLICY_CASES)
def test_wide_policy_head_matches_float64(algo, A, smoothing, n, M, table):
    """Butterfly (out_dim <= 8: SAC A = 4 is its last size) and per-output loop (A = 5, 17, 32: out_dim 64 = MAX_OUT, the
    largest shared-memory request); M across the 64-row CTA; stacked agents with per-agent td3_std / td3_c from the table
    (and without a table: the scalars); the xn obs copy from src_off, logp and the save layout [M][4][A]."""
    L = _lib()
    r = run_policy_head(L, algo, A, smoothing, n, M, table)
    td3, O, od = algo == "td3", r["O"], r["out_dim"]
    clamped = [0, 0]
    for a in range(n):
        rw = slice(a * M, (a + 1) * M)
        w3 = r["P"][a, :od * HID].view(od, HID)
        b3 = r["P"][a, od * HID:od * HID + od]
        ref = policy_head_ref(r["h2"][rw], w3, b3, r["eps"][rw], r["lo"], r["hi"], A, td3, bool(smoothing), r["stds"][a], r["cs"][a])
        tag = f"{algo} A={A} M={M} agent {a}"
        assert torch.equal(r["xn"][rw, :O], r["rows"][rw, r["src"]:r["src"] + O]), tag + ": xn obs copy"
        sat = ref.get("sat")
        check("wide_policy_head", tag + " action", r["xn"][rw, O:O + A], ref["act"], sat)
        check("wide_policy_head", tag + " tanh(head)", r["sv"][rw, 3], ref["th"])
        if td3:
            if smoothing:
                got = r["xn"][rw, O:O + A]
                clamped[0] += int((got == r["lo"]).sum())
                clamped[1] += int((got == r["hi"]).sum())
                assert torch.equal(r["eo"][rw], r["eps"][rw])
        else:
            check("wide_policy_head", tag + " logp", r["lp"][rw], ref["logp"], sat.any(1))
            assert torch.equal(r["sv"][rw, 0], r["eps"][rw]) and torch.equal(r["eo"][rw], r["eps"][rw])
            check("wide_policy_head", tag + " sigma", r["sv"][rw, 1], ref["sigma"])
            check("wide_policy_head", tag + " tanh(x)", r["sv"][rw, 2], ref["y"], sat)
    if td3 and smoothing and n * M * A >= 500:
        assert min(clamped) > 0, f"clamping at both ends not exercised: {clamped}"
    pad = torch.zeros_like(r["xn"], dtype=torch.bool)
    pad[:, O + A:] = True
    untouched(r["xn_f"], r["xn"], pad, "xn")
    untouched(r["lp_f"], what="logp")
    if td3:
        m = torch.zeros_like(r["sv"], dtype=torch.bool)
        m[:, :3] = True
        untouched(r["sv_f"], r["sv"], m, "save (TD3 uses slot 3 only)")
        if not smoothing:
            untouched(r["eo_f"], r["eo"], torch.ones_like(r["eo"], dtype=torch.bool), "eps_out (no noise drawn)")
        assert torch.isnan(r["lp"]).all()
    else:
        untouched(r["sv_f"], what="save")
        untouched(r["eo_f"], what="eps_out")


# ---- wide_q_head and tc_linear_q ------------------------------------------------------------------------------------------
def _q_inputs(g, n, M, rs):
    qn = torch.randn(2, n * M, device="cuda", generator=g) * 3.0
    tie = torch.rand(n * M, device="cuda", generator=g) < 0.1
    qn[1, tie] = qn[0, tie]
    rows = torch.randn(n * M, rs, device="cuda", generator=g)
    rows[:, 3] = (torch.rand(n * M, device="cuda", generator=g) < 0.3).float()  # done in {0, 1} (reward at column 2)
    logp = torch.randn(n * M, device="cuda", generator=g) * 2.0
    la = torch.zeros(n, 5, device="cuda")
    la[:, 0] = torch.tensor([-1.5, 0.3, -0.2][:n])
    return qn, rows, logp, la


def _wide_q(L, h2, w3, b3, q_out, qn, logp, rows, la, dz3, sq, targ, M, mode, rs, td3, bcq, gamma):
    q = L.WideQ()
    q.h2, q.w3, q.b3, q.q_out = L.ptr(h2), w3, b3, q_out.data_ptr()
    q.qn0, q.qn1, q.logp, q.rows, q.log_alpha = qn[0].data_ptr(), qn[1].data_ptr(), logp.data_ptr(), rows.data_ptr(), la.data_ptr()
    q.dz3, q.sq_part, q.targ_out = dz3.data_ptr(), sq.data_ptr(), L.ptr(targ)
    q.M, q.mode, q.row_stride, q.rd_off, q.td3, q.bcq_mix, q.gamma = M, mode, rs, 2, int(td3), int(bcq), gamma
    return q


def _check_q_outputs(kernel, tag, n, M, q_ref_of, qn, logp, la, rows, gammas, td3, bcq, mode, out, full):
    """q, TD target, dz3 (column 0 of [M][64]) and the per-8-row sq_part layout of each agent against float64."""
    qo, targ, dz3, sq = out
    P8 = (M + 7) // 8
    for a in range(n):
        rw = slice(a * M, (a + 1) * M)
        q = q_ref_of(a)
        check(kernel, f"{tag} agent {a} q", qo[rw], q)
        if not mode:
            continue
        t = q_target_ref(q, qn[0, rw], qn[1, rw], logp[rw], la[a, 0].double(), rows[rw, 2], rows[rw, 3], gammas[a], M, td3, bcq)
        check(kernel, f"{tag} agent {a} TD target", targ[rw], t["y"])
        check(kernel, f"{tag} agent {a} dLoss/dQ", dz3[rw, 0], t["dz"])
        parts = group_sum(R(torch.stack([t["sq"].v, t["dz"].v], 1), torch.stack([t["sq"].e, t["dz"].e], 1)), 8, 7)
        check(kernel, f"{tag} agent {a} sq_part", sq[a * P8:(a + 1) * P8], parts)
    qo_f, targ_f, dz3_f, sq_f = full
    m = torch.ones_like(dz3, dtype=torch.bool)
    if mode:
        m[:, 0] = False
    untouched(dz3_f, dz3, m, f"{kernel} dz3")
    untouched(qo_f, what=f"{kernel} q")
    untouched(targ_f, targ if not mode else None, torch.ones_like(targ, dtype=torch.bool) if not mode else None, f"{kernel} targ")
    untouched(sq_f, sq if not mode else None, torch.ones_like(sq, dtype=torch.bool) if not mode else None, f"{kernel} sq_part")


Q_CASES = [(mode, algo, bcq, 1, M, False) for mode in (0, 1) for algo in ("sac", "td3") for bcq in (0, 1) for M in (65,)] + [
    (1, "sac", 0, 1, M, False) for M in (1, 7, 8, 1000, 4097)] + [(1, "sac", 1, 3, 200, True), (1, "td3", 1, 3, 257, True),
                                                                 (1, "td3", 0, 3, 200, False), (0, "sac", 0, 3, 65, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode,algo,bcq,n,M,table", Q_CASES)
def test_wide_q_head_matches_float64(mode, algo, bcq, n, M, table):
    """wide_q_head: Q, and in mode 1 the TD target (done in {0, 1}, ties of the twin target Qs, BCQ mix, SAC's entropy
    term), dLoss/dQ and the per-CTA (8-row) partials, a ragged last group; stacked agents with per-agent gamma."""
    L = _lib()
    td3 = algo == "td3"
    g = torch.Generator(device="cuda").manual_seed(31 * M + n + mode)
    ps = HID + 4 + 60
    Pm = torch.randn(n, ps, device="cuda", generator=g) / 16.0
    Pm[:, HID] = torch.randn(n, device="cuda", generator=g)
    h2 = torch.relu(torch.randn(n * M, HID, device="cuda", generator=g))
    rs = 8
    qn, rows, logp, la = _q_inputs(g, n, M, rs)
    P8 = (M + 7) // 8
    full = [guarded(n * M), guarded(n * M), guarded(n * M, MAX_OUT), guarded(n * P8, 2)]
    out = [f[1] for f in full]
    hp, vals = hp_table(algo, n, gamma=[0.99, 0.9, 0.5][:n]) if table else (None, None)
    gammas = [f32(v["gamma"]) for v in vals] if table else [f32(0.97)] * n
    q = _wide_q(L, h2, Pm.data_ptr(), Pm.data_ptr() + 4 * HID, out[0], qn, logp, rows, la, out[2], out[3], out[1], M, mode, rs, td3, bcq, 0.97)
    stk = stack(L, n, 3, ps=ps, alpha=5, hp=hp) if (n > 1 or table) else None
    L.check(L.load().b2rl_wide_q_head(C.byref(q), None if stk is None else C.byref(stk), st()), "wide_q_head")
    torch.cuda.synchronize()
    q_ref = lambda a: r_dot(h2[a * M:(a + 1) * M], Pm[a, None, :HID], Pm[a, HID:HID + 1], 14)[:, 0]
    _check_q_outputs("wide_q_head", f"mode={mode} {algo} bcq={bcq} M={M}", n, M, q_ref, qn, logp, la, rows, gammas, td3, bcq, mode,
                     out, [f[0] for f in full])


def _layer_ref(X, W, b, gm, be, ln):
    z = X.double() @ W.double().T + b.double()
    if ln:
        z = (z - z.mean(1, keepdim=True)) / torch.sqrt(z.var(1, unbiased=False, keepdim=True) + 1e-5)
        z = z * gm.double() + be.double()
    return torch.relu(z)


TC3_TOL = 4e-6  # 3xTF32 hidden layer: fp32-level, of the layer's largest output (test_gpu_tc.py)


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,algo,bcq,ln,table", [(1, 65536, "sac", 0, 1, False), (1, 2056, "td3", 1, 1, False),
                                                   (1, 2048, "sac", 1, 0, False), (1, 2040, "td3", 0, 1, False),
                                                   (1, 8, "sac", 0, 1, False), (1, 65, "sac", 1, 1, False),
                                                   (3, 1000, "td3", 1, 1, True), (3, 2056, "sac", 0, 1, True)])
def test_tc_linear_q_and_critic_scalars_match_float64(n, M, algo, bcq, ln, table):
    """The critic head fused into tc_linear's epilogue (twin critics, mode 1; the target critics' form with H = NULL in
    mode 0), its sq_part fed into wide_critic_scalars: P = ceil(M / 8) partials = 1, 9, 125, 255, 256, 257 and 8 192 —
    across the 256-partial loop of wide_critic_scalars — and the loss / head-bias gradients of each agent against the
    float64 sums of the kernel's own partials (k above) and against the float64 loss."""
    L = _lib()
    lib = L.load()
    td3 = algo == "td3"
    g = torch.Generator(device="cuda").manual_seed(M + 7 * n + bcq)
    ps = 2 * (HID * HID + 4 * HID + 64)  # per agent: two critics [W | b | g | be | w3 | b3 ...]
    half = ps // 2
    Pm = torch.zeros(n, ps, device="cuda")
    for k in range(2):
        o = k * half
        Pm[:, o:o + HID * HID] = torch.randn(n, HID * HID, device="cuda", generator=g) / 16.0
        Pm[:, o + HID * HID:o + HID * HID + HID] = 0.1 * torch.randn(n, HID, device="cuda", generator=g)
        Pm[:, o + HID * HID + HID:o + HID * HID + 2 * HID] = 1.0 + 0.1 * torch.randn(n, HID, device="cuda", generator=g)
        Pm[:, o + HID * HID + 2 * HID:o + HID * HID + 3 * HID] = 0.1 * torch.randn(n, HID, device="cuda", generator=g)
        Pm[:, o + HID * HID + 3 * HID:o + HID * HID + 4 * HID] = torch.randn(n, HID, device="cuda", generator=g) / 16.0
        Pm[:, o + HID * HID + 4 * HID] = torch.randn(n, device="cuda", generator=g)
    X = torch.randn(n * M, HID, device="cuda", generator=g)
    rs = 8
    qn, rows, logp, la = _q_inputs(g, n, M, rs)
    P8 = (M + 7) // 8
    hp, vals = hp_table(algo, n, gamma=[0.99, 0.9, 0.5][:n]) if table else (None, None)
    gammas = [f32(v["gamma"]) for v in vals] if table else [f32(0.97)] * n
    stk = stack(L, n, 11, ps=ps, alpha=5, out=8, lo=ps, hp=hp) if (n > 1 or table) else None
    sp = None if stk is None else C.byref(stk)
    base = Pm.data_ptr()
    offs = lambda k: [base + 4 * (k * half + HID * HID + i * HID) for i in range(5)]  # b, g, be, w3, b3
    res = []
    for k in range(2):
        full = [guarded(n * M), guarded(n * M), guarded(n * M, MAX_OUT), guarded(n * P8, 2)]
        out = [f[1] for f in full]
        W = base + 4 * k * half
        ob, og, obe, ow3, ob3 = offs(k)
        q = _wide_q(L, None, ow3, ob3, out[0], qn, logp, rows, la, out[2], out[3], out[1], M, 1, rs, td3, bcq, 0.97)
        XH = torch.empty(n * M, HID, device="cuda")
        stat = torch.empty(n * M, 2, device="cuda")
        L.check(lib.b2rl_tc_linear_q(X.data_ptr(), HID, M, W, W, ob, og if ln else None, obe if ln else None, ln, None, XH.data_ptr(),
                                     stat.data_ptr(), C.byref(q), sp, st()), "tc_linear_q")
        res.append((out, full))
    # mode 0 (the target critics): q only, h2 not stored
    f0 = [guarded(n * M), guarded(n * M), guarded(n * M, MAX_OUT), guarded(n * P8, 2)]
    q0 = _wide_q(L, None, offs(0)[3], offs(0)[4], f0[0][1], qn, logp, rows, la, f0[2][1], f0[3][1], f0[1][1], M, 0, rs, td3, bcq, 0.97)
    L.check(lib.b2rl_tc_linear_q(X.data_ptr(), HID, M, base, base, offs(0)[0], offs(0)[1] if ln else None, offs(0)[2] if ln else None,
                                 ln, None, None, None, C.byref(q0), sp, st()), "tc_linear_q mode 0")
    # the twin critics' partials -> qf_loss and the head-bias gradients
    G_f, G = guarded(n, ps)
    o_f, outv = guarded(n, 8)
    (o0, _), (o1, _) = res
    L.check(lib.b2rl_wide_critic_scalars(o0[3].data_ptr(), o1[3].data_ptr(), P8, None, None, M, G.data_ptr(), HID * HID + 4 * HID,
                                         half + HID * HID + 4 * HID, outv.data_ptr(), sp, st()), "wide_critic_scalars")
    torch.cuda.synchronize()
    tag = f"{algo} bcq={bcq} ln={ln} M={M} n={n}"
    refs = []
    for k in range(2):
        o = k * half

        def q_ref(a, o=o):
            rw = slice(a * M, (a + 1) * M)
            h = _layer_ref(X[rw], Pm[a, o:o + HID * HID].view(HID, HID), *[Pm[a, o + HID * HID + i * HID:o + HID * HID + (i + 1) * HID]
                                                                       for i in range(3)], ln)
            w3 = Pm[a, o + HID * HID + 3 * HID:o + HID * HID + 4 * HID].double()
            e_h = TC3_TOL * float(h.abs().max())
            qv = h @ w3 + float(Pm[a, o + HID * HID + 4 * HID])
            return R(qv, e_h * float(w3.abs().sum()) + gam(258) * (h.abs() @ w3.abs() + abs(float(Pm[a, o + HID * HID + 4 * HID]))))

        out, full = res[k]
        _check_q_outputs("tc_linear_q", f"{tag} critic {k}", n, M, q_ref, qn, logp, la, rows, gammas, td3, bcq, 1, out, [f[0] for f in full])
        refs.append(q_ref)
    _check_q_outputs("tc_linear_q", f"{tag} mode 0", n, M, refs[0], qn, logp, la, rows, gammas, td3, bcq, 0, [f[1] for f in f0],
                     [f[0] for f in f0])
    owned = torch.zeros(n, ps, dtype=torch.bool, device="cuda")
    owned[:, [HID * HID + 4 * HID, half + HID * HID + 4 * HID]] = True
    for a in range(n):
        s0, s1 = o0[3][a * P8:(a + 1) * P8], o1[3][a * P8:(a + 1) * P8]
        loss, d0, d1 = critic_scalars_ref(s0, s1, M)
        check("wide_critic_scalars", f"{tag} agent {a} qf_loss (P={P8})", outv[a, L.OUT_QF_LOSS], loss)
        check("wide_critic_scalars", f"{tag} agent {a} d b3_0", G[a, HID * HID + 4 * HID], d0)
        check("wide_critic_scalars", f"{tag} agent {a} d b3_1", G[a, half + HID * HID + 4 * HID], d1)
        # and the whole chain against the float64 loss: sum of both critics' mean squared TD errors
        rw = slice(a * M, (a + 1) * M)
        tot = None
        for k in range(2):
            t = q_target_ref(refs[k](a), qn[0, rw], qn[1, rw], logp[rw], la[a, 0].double(), rows[rw, 2], rows[rw, 3], gammas[a], M,
                             td3, bcq)
            s = r_sum(t["sq"], 0, 3 + 2 * math.ceil(P8 / 256) + min(P8, 256))
            tot = s if tot is None else tot + s
        check("wide_critic_scalars", f"{tag} agent {a} qf_loss vs the float64 loss", outv[a, L.OUT_QF_LOSS], tot / R(float(M)))
    untouched(G_f, G, ~owned, "G (critic scalars)")
    m = torch.ones(n, 8, dtype=torch.bool, device="cuda")
    m[:, L.OUT_QF_LOSS] = False
    untouched(o_f, outv, m, "out (critic scalars)")


# ---- wide_colsum_multi / wide_colsum --------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 63, 64, 65, 512, 2048])
@pytest.mark.parametrize("n_jobs,n", [(1, 1), (8, 3)])
def test_wide_colsum_matches_float64(P, n_jobs, n):
    """Column sums of P per-CTA partials: P = 64 switches from 8 to 32 slices (256 -> 1 024 threads); jobs with and without
    LayerNorm (their off_g / off_be entries must stay untouched), stacked agents; every job of the multi launch bitwise
    equal to a wide_colsum launch of its own."""
    L = _lib()
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(P + 100 * n_jobs)
    parts = [torch.randn(n, P, 3, HID, device="cuda", generator=g) * (1 + j) for j in range(n_jobs)]
    lns = [(j % 3) != 1 for j in range(n_jobs)]
    ps = 3 * HID * n_jobs + 40
    offs = [(3 * HID * j + 8, 3 * HID * j + 8 + HID, 3 * HID * j + 8 + 2 * HID) for j in range(n_jobs)]
    arr = (L.ColsumJob * n_jobs)()
    for a, p, (ob, og, obe), ln in zip(arr, parts, offs, lns):
        a.part, a.off_b, a.off_g, a.off_be, a.layer_norm = p.data_ptr(), ob, og, obe, int(ln)
    stk = stack(L, n, 2, ps=ps) if n > 1 else None
    sp = None if stk is None else C.byref(stk)
    G_f, G = guarded(n, ps)
    L.check(lib.b2rl_wide_colsum_multi(arr, n_jobs, P, G.data_ptr(), sp, st()), "wide_colsum_multi")
    singles = []
    for p, (ob, og, obe), ln in zip(parts, offs, lns):
        Gs_f, Gs = guarded(n, ps)
        L.check(lib.b2rl_wide_colsum(p.data_ptr(), P, Gs.data_ptr(), ob, og, obe, int(ln), sp, st()), "wide_colsum")
        singles.append((Gs_f, Gs))
    torch.cuda.synchronize()
    owned = torch.zeros(n, ps, dtype=torch.bool, device="cuda")
    for j, (p, (ob, og, obe), ln) in enumerate(zip(parts, offs, lns)):
        nv = 3 if ln else 1
        own_j = torch.zeros_like(owned)
        for a in range(n):
            ref = colsum_ref(p[a], colsum_k(P))
            for v, off in enumerate((ob, og, obe)[:nv]):
                check("wide_colsum", f"P={P} job {j} agent {a} vector {v}", G[a, off:off + HID], ref[v])
                own_j[a, off:off + HID] = True
        owned |= own_j
        Gs_f, Gs = singles[j]
        assert torch.equal(Gs[own_j], G[own_j]), f"job {j}: multi != single launch"
        untouched(Gs_f, Gs, ~own_j, f"wide_colsum job {j}")
    untouched(G_f, G, ~owned, "wide_colsum_multi")


# ---- actor step kernels ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("algo,n,M", [("sac", 1, 1), ("sac", 1, 255), ("sac", 1, 256), ("sac", 1, 257), ("sac", 1, 4097),
                                      ("td3", 1, 1000), ("sac", 3, 600), ("td3", 3, 257)])
def test_wide_actor_loss_and_scalars_match_float64(algo, n, M):
    """wide_actor_loss (exact ties: the whole gradient to critic 0; TD3 with q1 = NULL), then wide_actor_scalars on its
    partials (P = ceil(M / 256) = 1, 2, 17, 3 ...) and on head-bias partials: loss, mean log-prob, alpha and G[off_b3 + t]."""
    L = _lib()
    lib = L.load()
    td3 = algo == "td3"
    g = torch.Generator(device="cuda").manual_seed(M + n)
    q = torch.randn(2, n * M, device="cuda", generator=g) * 5.0
    tie = torch.rand(n * M, device="cuda", generator=g) < 0.2
    q[1, tie] = q[0, tie]
    logp = torch.randn(n * M, device="cuda", generator=g) * 3.0
    la = torch.full((n, 8), float("nan"), device="cuda")
    la[:, 0] = torch.tensor([-1.0, 0.5, -2.0][:n])
    P = (M + 255) // 256
    dz0_f, dz0 = guarded(n * M, MAX_OUT)
    dz1_f, dz1 = guarded(n * M, MAX_OUT)
    ps_f, part_s = guarded(n * P, 2)
    A = 5
    out_dim = A if td3 else 2 * A
    part_du = torch.randn(n * P, MAX_OUT, device="cuda", generator=g)
    part_du[:, out_dim:] = float("nan")  # (columns past the head never exist in a real step)
    gps = 3 * MAX_OUT + 16
    G_f, G = guarded(n, gps)
    o_f, outv = guarded(n, 8)
    stk = stack(L, n, 9, ps=gps, alpha=8, out=8) if n > 1 else None
    sp = None if stk is None else C.byref(stk)
    L.check(lib.b2rl_wide_actor_loss(q[0].data_ptr(), None if td3 else q[1].data_ptr(), None if td3 else logp.data_ptr(),
                                     None if td3 else la.data_ptr(), int(td3), M, dz0.data_ptr(), None if td3 else dz1.data_ptr(),
                                     part_s.data_ptr(), sp, st()), "wide_actor_loss")
    off_b3 = MAX_OUT + 5
    L.check(lib.b2rl_wide_actor_scalars(part_s.data_ptr(), part_du.data_ptr(), P, M, out_dim, int(td3), None if td3 else la.data_ptr(),
                                        G.data_ptr(), off_b3, outv.data_ptr(), sp, st()), "wide_actor_scalars")
    torch.cuda.synchronize()
    for a in range(n):
        rw = slice(a * M, (a + 1) * M)
        ref = actor_loss_ref(q[0, rw], None if td3 else q[1, rw], logp[rw], la[a, 0].double(), td3, M)
        tag = f"{algo} M={M} agent {a}"
        check("wide_actor_loss", tag + " dLoss/dQ0", dz0[rw, 0], ref["d0"])
        if not td3:
            check("wide_actor_loss", tag + " dLoss/dQ1", dz1[rw, 0], ref["d1"])
            t = tie[rw]
            assert bool((dz1[rw, 0][t] == 0).all()) and bool((dz0[rw, 0][t] != 0).all()), tag + ": ties must go to critic 0"
        s = group_sum(R(torch.stack([ref["loss"].v, ref["lp"].v], 1), torch.stack([ref["loss"].e, ref["lp"].e], 1)), 256, 12)
        check("wide_actor_loss", tag + " partials", part_s[a * P:(a + 1) * P], s)
        # wide_actor_scalars, from the kernel's own partials
        ps_a = part_s[a * P:(a + 1) * P].double()
        check("wide_actor_scalars", tag + f" actor loss (P={P})", outv[a, L.OUT_ACTOR_LOSS], r_sum(R(ps_a[:, 0]), 0, P) / R(float(M)))
        check("wide_actor_scalars", tag + " mean logpi", outv[a, L.OUT_LOGPI_MEAN], r_sum(R(ps_a[:, 1]), 0, P) / R(float(M)))
        check("wide_actor_scalars", tag + " d head.bias", G[a, off_b3:off_b3 + out_dim],
              r_sum(R(part_du[a * P:(a + 1) * P, :out_dim]), 0, P))
        if not td3:
            check("wide_actor_scalars", tag + " alpha", outv[a, L.OUT_ALPHA], r_exp(R(la[a, 0])))
    m = torch.ones_like(dz0, dtype=torch.bool)
    m[:, 0] = False
    untouched(dz0_f, dz0, m, "dzq0")
    untouched(dz1_f, dz1, m if not td3 else torch.ones_like(m), "dzq1")
    untouched(ps_f, what="part_s")
    owned = torch.zeros(n, gps, dtype=torch.bool, device="cuda")
    owned[:, off_b3:off_b3 + out_dim] = True
    untouched(G_f, G, ~owned, "G (actor scalars)")
    mo = torch.ones(n, 8, dtype=torch.bool, device="cuda")
    mo[:, [L.OUT_ACTOR_LOSS, L.OUT_LOGPI_MEAN] + ([] if td3 else [L.OUT_ALPHA])] = False
    untouched(o_f, outv, mo, "out (actor scalars)")


@pytest.mark.gpu
@pytest.mark.parametrize("A", [1, 3, 8, 17, 32])
@pytest.mark.parametrize("n,M", [(1, 63), (1, 64), (1, 65), (1, 1000), (3, 200)])
def test_wide_dqda_matches_float64(A, n, M):
    """dQ/da = dz1 . w1t[O + a][:] per row: M across the 64-row CTA and its one-row-ahead load; stacked agents."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(A * 1000 + M + n)
    ps = A * HID + 36
    W = torch.randn(n, ps, device="cuda", generator=g) / 16.0
    dz1 = torch.randn(n * M, HID, device="cuda", generator=g)
    o_f, out = guarded(n * M, A)
    stk = stack(L, n, 1, ps=ps) if n > 1 else None
    L.check(L.load().b2rl_wide_dqda(dz1.data_ptr(), W.data_ptr(), A, M, out.data_ptr(), None if stk is None else C.byref(stk), st()),
            "wide_dqda")
    torch.cuda.synchronize()
    for a in range(n):
        rw = slice(a * M, (a + 1) * M)
        check("wide_dqda", f"A={A} M={M} agent {a}", out[rw], r_dot(dz1[rw], W[a, :A * HID].view(A, HID), torch.zeros(A, device="cuda"), 13))
    untouched(o_f, what="dqda")


def _saturated_save(g, N, A):
    """Hand-made [N][4][A] save rows: y = tanh(x) within a few ulp of +-1 (and exactly +-1), th near +-1, sigma over its range."""
    sv = torch.empty(N, 4, A, device="cuda")
    sv[:, 0] = torch.randn(N, A, device="cuda", generator=g)
    sv[:, 1] = torch.exp(-5.0 + 7.0 * torch.rand(N, A, device="cuda", generator=g))
    k = torch.randint(0, 40, (N, A), device="cuda", generator=g).float()
    y = 1.0 - k * 2.0 ** -24
    y = torch.where(torch.rand(N, A, device="cuda", generator=g) < 0.3, 1.0 - 1e-4 * torch.rand(N, A, device="cuda", generator=g), y)
    sgn = torch.where(torch.rand(N, A, device="cuda", generator=g) < 0.5, -1.0, 1.0)
    sv[:, 2] = sgn * y
    sv[:, 3] = torch.tanh(3.0 * torch.randn(N, A, device="cuda", generator=g))
    return sv


@pytest.mark.gpu
@pytest.mark.parametrize("algo,A,n,M,source", [("sac", 17, 1, 257, "policy"), ("sac", 32, 1, 257, "policy"), ("sac", 17, 3, 300, "policy"),
                                               ("sac", 17, 1, 513, "saturated"), ("sac", 32, 3, 200, "saturated"),
                                               ("td3", 17, 1, 257, "policy"), ("td3", 5, 3, 300, "saturated")])
def test_wide_actor_head_bwd_matches_float64(algo, A, n, M, source):
    """Backward through the action head: SAC at 34 and 64 outputs, TD3; save taken from wide_policy_head itself and from
    hand-made near-saturated values (where fp32 1 - y^2 cancels); du [M][64] and the per-CTA part_du [P][64]."""
    L = _lib()
    lib = L.load()
    td3 = algo == "td3"
    g = torch.Generator(device="cuda").manual_seed(A * 7 + M + n)
    out_dim = A if td3 else 2 * A
    if source == "policy":
        r = run_policy_head(L, algo, A, 0, n, M, False, seed=5)
        save, lo, hi = r["sv"].clone(), r["lo"], r["hi"]
        if td3:
            save[:, :3] = 0.0
    else:
        save = _saturated_save(g, n * M, A)
        lo = -0.5 - torch.rand(A, device="cuda", generator=g)
        hi = 0.2 + 1.5 * torch.rand(A, device="cuda", generator=g)
    dq = torch.randn(2, n * M, A, device="cuda", generator=g)
    la = torch.zeros(n, 5, device="cuda")
    la[:, 0] = torch.tensor([-1.2, 0.4, -3.0][:n])
    P = (M + 255) // 256
    du_f, du = guarded(n * M, MAX_OUT)
    pd_f, pdu = guarded(n * P, MAX_OUT)
    stk = stack(L, n, 4, alpha=5) if n > 1 else None
    L.check(lib.b2rl_wide_actor_head_bwd(dq[0].data_ptr(), None if td3 else dq[1].data_ptr(), save.data_ptr(), lo.data_ptr(), hi.data_ptr(),
                                         None if td3 else la.data_ptr(), int(td3), A, M, du.data_ptr(), pdu.data_ptr(),
                                         None if stk is None else C.byref(stk), st()), "wide_actor_head_bwd")
    torch.cuda.synchronize()
    for a in range(n):
        rw = slice(a * M, (a + 1) * M)
        ref = head_bwd_ref(dq[0, rw], None if td3 else dq[1, rw], save[rw], lo, hi, la[a, 0], td3, A, M)
        tag = f"{algo} A={A} M={M} {source} agent {a}"
        check("wide_actor_head_bwd", tag + " du", du[rw, :out_dim], ref["du"], ref["sat"])
        check("wide_actor_head_bwd", tag + " part_du", pdu[a * P:(a + 1) * P, :out_dim], group_sum(ref["du"], 256, 12))
    m = torch.zeros_like(du, dtype=torch.bool)
    m[:, out_dim:] = True
    untouched(du_f, du, m, "du")
    mp = torch.zeros_like(pdu, dtype=torch.bool)
    mp[:, out_dim:] = True
    untouched(pd_f, pdu, mp, "part_du")


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,table", [(1, 1, False), (1, 255, False), (1, 4095, False), (1, 4096, False), (1, 4097, False),
                                       (1, 65536, False), (3, 5000, True), (3, 5000, False)])
def test_wide_alpha_grad_matches_float64(n, M, table):
    """alpha_state[1] <- alpha * mean(-logpi - targ_ent): M across the 4 096-row pass of the sixteen-loads loop and at
    65 536 (16 passes); per-agent targ_ent from the table against the scalar."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(M + n)
    lp = torch.randn(n * M, device="cuda", generator=g) * 2.0 + 1.0
    as_f, ast = guarded(n, 6)
    ast[:, 0] = torch.tensor([-1.0, 0.2, -0.7][:n])
    hp, vals = hp_table("sac", n, targ_ent=[-3.0, -1.5, 0.25][:n]) if table else (None, None)
    tes = [f32(v["targ_ent"]) for v in vals] if table else [f32(-3.0)] * n
    stk = stack(L, n, 0, alpha=6, hp=hp) if (n > 1 or table) else None
    L.check(L.load().b2rl_wide_alpha_grad(lp.data_ptr(), M, -3.0, ast.data_ptr(), None if stk is None else C.byref(stk), st()),
            "wide_alpha_grad")
    torch.cuda.synchronize()
    for a in range(n):
        check("wide_alpha_grad", f"M={M} agent {a} targ_ent={tes[a]}", ast[a, 1], alpha_grad_ref(lp[a * M:(a + 1) * M], ast[a, 0], tes[a]))
    m = torch.ones(n, 6, dtype=torch.bool, device="cuda")
    m[:, :2] = False
    untouched(as_f, ast, m, "alpha state")


@pytest.mark.gpu
def test_report_worst_ratios():
    """(runs last in this module) the worst deviation / bound ratio of each kernel over the tests above."""
    for k, v in sorted(WORST.items()):
        print(f"worst dev/bound {k:22s} {v:.3f}")


# ---- the bounds have teeth (no GPU) --------------------------------------------------------------------------------------
def _teeth(name, wrong, ref: R, at_least=10.0):
    ratio = float(((wrong.double() - ref.v).abs() / (WIDEN * ref.e + FLOOR)).max())
    assert ratio >= at_least, f"{name}: the bound accepts this mistake (worst ratio {ratio:.2f})"
    return ratio


def _fp32_within(name, got, ref: R):
    ratio = float(((got.double() - ref.v).abs() / (WIDEN * ref.e + FLOOR)).max())
    assert ratio <= 1.0, f"{name}: an fp32 evaluation exceeds its bound ({ratio:.2f})"


def test_bounds_have_teeth():
    """At small shapes on the CPU: each float64 reference's bound rejects, at least tenfold, plausible mistakes applied to
    that reference — and accepts an fp32 evaluation of the same operation in another summation order."""
    g = torch.Generator().manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g)
    # column sums / critic scalars / actor scalars: one partial dropped, or counted twice
    part = rn(65, 3, HID)
    ref = colsum_ref(part, colsum_k(65))
    _fp32_within("colsum", part.sum(0), ref)
    _teeth("colsum, partial dropped", part[1:].double().sum(0), ref)
    _teeth("colsum, partial counted twice", part.double().sum(0) + part[7].double(), ref)
    sq0, sq1 = rn(300, 2).abs(), rn(300, 2).abs()
    loss, d0, _ = critic_scalars_ref(sq0, sq1, 2400)
    _fp32_within("critic scalars", (sq0[:, 0] + sq1[:, 0]).sum() / 2400, loss)
    _teeth("critic scalars, partial dropped", (sq0[1:, 0].double().sum() + sq1[:, 0].double().sum()) / 2400, loss)
    _teeth("critic scalars (d b3), partial counted twice", sq0[:, 1].double().sum() + sq0[299, 1].double(), d0)
    pdu = rn(3, 10)
    ref = r_sum(R(pdu), 0, 3)
    _teeth("actor scalars, partial counted twice", pdu.double().sum(0) + pdu[2].double(), ref)
    # the critic head (two stacked agents): the neighbour's parameters or rows, 2 / M over all agents' rows
    M, n = 40, 2
    h2 = torch.relu(rn(n * M, HID))
    w3 = rn(n, 1, HID) / 16.0
    b3 = rn(n, 1)
    qn, lp, r = rn(2, n * M) * 3, rn(n * M), rn(n * M)
    d = (torch.rand(n * M, generator=g) < 0.3).float()
    ref_q = r_dot(h2[:M], w3[0], b3[0], 14)[:, 0]
    _fp32_within("q head", (h2[:M] @ w3[0].T + b3[0])[:, 0], ref_q)
    _teeth("q head, neighbour's w3", (h2[:M].double() @ w3[1].double().T + b3[1].double())[:, 0], ref_q)
    _teeth("q head, neighbour's rows", (h2[M:].double() @ w3[0].double().T + b3[0].double())[:, 0], ref_q)
    t = q_target_ref(ref_q, qn[0, :M], qn[1, :M], lp[:M], -1.0, r[:M], d[:M], 0.99, M, False, True)
    tw = q_target_ref(ref_q, qn[0, :M], qn[1, :M], lp[:M], -1.0, r[:M], d[:M], 0.99, n * M, False, True)
    _teeth("dLoss/dQ, 2 / M over all agents' rows", tw["dz"].v, t["dz"])
    tn = q_target_ref(ref_q, qn[0, M:], qn[1, M:], lp[M:], -1.0, r[M:], d[M:], 0.99, M, False, True)
    _teeth("TD target, neighbour's rows", tn["y"].v, t["y"])
    # actor loss: the tie gradient sent to critic 1
    q0, q1 = rn(M), rn(M)
    q1[::3] = q0[::3]
    ref = actor_loss_ref(q0, q1, lp[:M], -1.0, False, M)
    wrong = torch.where(q0 < q1, -1.0 / M, 0.0)  # (strict <: ties to critic 1)
    _teeth("actor loss, ties to critic 1", wrong, ref["d0"])
    # policy head: the neighbour's parameters; dQ/da: the neighbour's w1t rows; head backward: the neighbour's rows
    A = 3
    w = rn(n, 2 * A, HID) / 8.0
    bb = rn(n, 2 * A) * 0.3
    eps = rn(M, A)
    lo, hi = -torch.ones(A), torch.ones(A) * 0.5
    ref = policy_head_ref(h2[:M], w[0], bb[0], eps, lo, hi, A, False)
    nb = policy_head_ref(h2[:M], w[1], bb[1], eps, lo, hi, A, False)
    _teeth("policy head (action), neighbour's w3", nb["act"].v, ref["act"])
    _teeth("policy head (logp), neighbour's w3", nb["logp"].v, ref["logp"])
    dz1 = rn(n * M, HID)
    w1a = rn(n, A, HID) / 16.0
    ref = r_dot(dz1[:M], w1a[0], torch.zeros(A), 13)
    _fp32_within("dqda", dz1[:M] @ w1a[0].T, ref)
    _teeth("dqda, neighbour's w1t", dz1[:M].double() @ w1a[1].double().T, ref)
    sv = torch.stack([eps, torch.exp(rn(M, A)), torch.tanh(rn(M, A) * 2), torch.tanh(rn(M, A))], 1)
    dq = rn(n * M, A)
    ref = head_bwd_ref(dq[:M], dq[:M], sv, lo, hi, torch.tensor(-1.0), False, A, M)
    wrong = head_bwd_ref(dq[M:], dq[M:], sv, lo, hi, torch.tensor(-1.0), False, A, M)
    _teeth("head backward, neighbour's rows", wrong["du"].v, ref["du"])
    # temperature: another agent's targ_ent
    lp2 = rn(5000) * 2 + 1
    ref = alpha_grad_ref(lp2, -1.0, -3.0)
    _fp32_within("alpha grad", torch.exp(torch.tensor(-1.0)) * (-lp2 - f32(-3.0)).sum() / 5000, ref)
    _teeth("alpha grad, another agent's targ_ent", alpha_grad_ref(lp2, -1.0, -1.5).v, ref)
