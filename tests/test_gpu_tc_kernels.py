"""The tcgen05 kernels (csrc/tc_linear.cu, csrc/tc_wgrad.cu) and the wide path's FFMA first layer / LayerNorm backward
(csrc/wide.cu) against a float64 restatement, element by element, at the sizes where their tile walkers, vector-set swaps,
batch splits and reductions change.

The kernels are called directly through _lib with fp32 inputs; the references are computed in float64 (on the GPU) from
those same fp32 values, with u = 2^-24 and gamma_k as in tests/helpers.py.

Tensor-core products. The kernels' own comments (tc_linear.cu:26-29, :37-45) describe the tensor core as reading fp32
operands as TF32 by truncation and accumulating in fp32. The reference emulates the operands exactly:
    hi(x) = x & 0xFFFFE000 (the truncation),   lo'(x) = hi(x - hi(x)) (the stored lo part, truncated again on reading),
    TF32:   sum hi(a) hi(b);   3xTF32: sum hi(a) hi(b) + lo'(a) hi(b) + hi(a) lo'(b).
Products of TF32 values are exact in float64, so what remains between kernel and reference is the fp32 accumulation.

Accumulation bound. One tcgen05.mma kind::tf32 (K = 8) adds its 8 products to the accumulator element. Assumed model
(NVIDIA does not document it; this follows the published measurements of earlier NVIDIA tensor cores): the 9 terms
(accumulator and 8 exact products) are aligned to the exponent E of the largest, each truncated below the 24th significant
bit of that alignment, summed, and the sum truncated to fp32. With no guard bits at all, each of the 8 aligned terms other
than the largest loses less than 2^(E-23) <= 2u max|t|, and the final truncation less than one ulp <= 2u |result|; so
    |error of one instruction| <= c u (|acc| + sum |its 8 products|),   c = 8 * 2 + 2 = 18,
added up over the instructions that accumulate into the element, in the kernel's issue order (|acc| is the exact partial
sum before the instruction): K/8 instructions for TF32, 3K/8 for 3xTF32, ordered per 32-wide k-slab as the issuer loops do
(tc_linear.cu:384-396: PREC 1 hi.hi, hi.lo' per k, then lo'.hi per k; PREC 2 and tc_wgrad.cu:240-249: hi.hi per k, then
lo'.hi, hi.lo' per k). Instructions whose products are all zero (k beyond K) leave the accumulator as it is. Any guard bits
the hardware keeps make the true error smaller; the measured ratios (DESIGN.md §4) are what validate the model. A second,
looser check compares with the TRUE float64 product, adding the truncation error per term (2^-9 + 2^-20 for TF32, 3 2^-20
for 3xTF32) to the accumulation bound: a check of the emulation itself.

tc_wgrad: each batch split accumulates in TMEM as above (its own instruction chain); the reduce kernel adds the slices in
its fixed order (tc_wgrad.cu:372-391): warp w adds slices w, w + 8, w + 16, ... in sequence, then the 8 warps' sums are
added in warp order — restated operation by operation with class R. The direct path (stacked, one split) has no reduce.

Later stages are checked from the kernel's own stored input, as in test_gpu_fused_kernels.py:
  - statistics (mean, rstd): the kernel's shifted one-pass formulas restated with R on the emulated z with its bound (first-
    order sensitivity), in the order the kernel combines them (tc_linear.cu:494-527; EPW = 8: two halves of 128 columns
    combined as at :519-521). The shift cancels exactly from mean and variance, so it is taken as exact;
  - x-hat from z and the kernel's own stat; H from the kernel's own x-hat (one fma and a ReLU);
  - backward: the ReLU mask fma(x-hat, gamma, beta) > 0 has the sign of the exact value, so it is exact in float64 and no
    row is set aside; dz1 under R over the two column halves (chains of 128); each tile's three partials separately — the
    sum of dz from the kernel's own DZ1, the other two from the reference dn under its bound — with k = 31 + 2 for
    tile_colsum and the (w0 + w1) + (w2 + w3) combine (:741);
  - wide_first: a sequential FMA chain over K, then the two-pass LayerNorm (wide.cu:53-117: chains of 8 and 13);
  - wide_ln_bwd: chains of n_out (head), 13 (row sums), 16 rows per warp + 8 warps (partials).

Every output lies in a NaN guard band; parameter tensors are NaN between agents; X is NaN between K and ldx; tc_wgrad's
scratch is NaN before each launch. Each owned element must come back finite; everything else must still be NaN, bitwise.
The worst deviation / bound ratio of each kernel and output is printed by test_report_worst_ratios.

test_bounds_have_teeth (no GPU) shows each bound rejects, at least tenfold, the mistakes the kernels could plausibly make.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests.helpers import FLOOR, WIDEN, R, U, gam, guarded, r_sum, untouched

HID, MAX_OUT = 256, 64
C_MMA = 18                               # see the module docstring
T_TRUE = {"tf32": 2.0 ** -9 + 2.0 ** -20, "x3w": 3 * 2.0 ** -20, "x3": 3 * 2.0 ** -20}
LN_EPS = float(np.float32(1e-5))
PAD = 4                                  # NaN floats after each agent's parameter block
WORST: dict = {}


# ---- emulated tensor core ------------------------------------------------------------------------------------------------
def hi(x):
    """The TF32 truncation: the low 13 mantissa bits cleared (fp32 in, fp32 out)."""
    return (x.contiguous().view(torch.int32) & -8192).view(torch.float32)


def lo3(x):
    return hi(x - hi(x))


def mma_acc(A, B, prec):
    """A [..., M, K] . B [..., N, K]^T as the tensor core accumulates it. prec: 'tf32', 'x3w' (PREC 1: the weights' lo
    parts from a mirror) or 'x3' (PREC 2 / tc_wgrad: lo parts made in shared memory). Returns (emulated value R with its
    accumulation bound, the true float64 product, sum |a||b|)."""
    K = A.shape[-1]
    ah, bh = hi(A).double(), hi(B).double()
    if prec != "tf32":
        al, bl = lo3(A).double(), lo3(B).double()
    acc = torch.zeros(*A.shape[:-1], B.shape[-2], dtype=torch.float64, device=A.device)
    e = torch.zeros_like(acc)
    for k0 in range(0, K, 32):
        ks = [slice(k, min(k + 8, K)) for k in range(k0, min(k0 + 32, K), 8)]
        if prec == "tf32":
            ins = [(ah, bh, s) for s in ks]
        elif prec == "x3w":
            ins = [q for s in ks for q in ((ah, bh, s), (ah, bl, s))] + [(al, bh, s) for s in ks]
        else:
            ins = [(ah, bh, s) for s in ks] + [q for s in ks for q in ((al, bh, s), (ah, bl, s))]
        for a, b, s in ins:
            a_, b_ = a[..., s], b[..., s]
            e += C_MMA * U * (acc.abs() + a_.abs() @ b_.abs().mT)
            acc += a_ @ b_.mT
    Ad, Bd = A.double(), B.double()
    return R(acc, e), Ad @ Bd.mT, Ad.abs() @ Bd.abs().mT


def r_sqrt(a: R) -> R:
    v = torch.sqrt(a.v)
    return R(v, a.e / (2 * v) + U * v)


def r_relu(a: R) -> R:  # (1-Lipschitz, exact in fp32)
    return R(a.v.clamp_min(0), a.e)


def ln_stats(z: R, epw8: bool):
    """The epilogue's shifted one-pass LayerNorm statistics of z [..., 256] (tc_linear.cu:494-527) under R."""
    def part(zh):
        sh = R(zh.v[..., :32].mean(-1, keepdim=True))  # (the shift cancels from mean and variance: exact)
        d = zh - sh
        return sh, r_sum(d, -1, zh.v.shape[-1] - 1), r_sum(d * d, -1, zh.v.shape[-1] - 1)
    if epw8:
        NH = 128.0
        (sh0, a0, q0), (sh1, a1, q1) = part(z[..., :128]), part(z[..., 128:])
        sh0, sh1 = sh0[..., 0], sh1[..., 0]
        mean = ((NH * sh0 + a0) + (NH * sh1 + a1)) * (1.0 / HID)
        e0, e1 = mean - sh0, mean - sh1
        var = ((q0 - 2.0 * e0 * a0 + NH * e0 * e0) + (q1 - 2.0 * e1 * a1 + NH * e1 * e1)) * (1.0 / HID)
    else:
        sh, s1, s2 = part(z)
        m = s1 * (1.0 / HID)
        mean = sh[..., 0] + m
        var = s2 * (1.0 / HID) - m * m
    return mean, R(1.0) / r_sqrt(var + LN_EPS)


def fwd_ref(acc: R, b, g, be, ln, relu, epw8, stat=None, xh=None):
    """The forward epilogue from the accumulator (R) and the per-agent vectors [n, 256]: dict of R references for
    mean / rstd / x-hat (or pre-activation) / H; stat and xh, when given, are the kernel's own stored values."""
    z = acc + R(b[:, None, :])
    out = {}
    if ln:
        mean, rstd = ln_stats(z, epw8)
        out["mean"], out["rstd"] = mean, rstd
        mk, rk = (mean, rstd) if stat is None else (R(stat[..., 0]), R(stat[..., 1]))
        out["xh"] = (z - R(mk.v[..., None], mk.e[..., None])) * R(rk.v[..., None], rk.e[..., None])
        x = out["xh"] if xh is None else R(xh)
        y = x * R(g[:, None, :]) + R(be[:, None, :])
    else:
        out["xh"] = z
        y = z if xh is None else R(xh)
    out["h"] = r_relu(y) if relu else y
    return out


def check(kernel, what, got, ref: R, true=None):
    """|got - ref.v| <= ref.e (widened), element-wise; true = (float64 value, allowance): the looser check against the true
    product."""
    got = got.detach()
    assert torch.isfinite(got).all(), f"{kernel} {what}: an owned element was not written (or is not finite)"
    dev = (got.double() - ref.v).abs()
    r = float((dev / (WIDEN * ref.e + FLOOR)).max())
    key = f"{kernel} {what.split(':')[0]}"
    WORST[key] = max(WORST.get(key, 0.0), r)
    msg = f"{kernel} {what}: worst dev/bound {r:.3f}"
    if true is not None:
        rt = float(((got.double() - true[0]).abs() / (WIDEN * true[1] + FLOOR)).max())
        msg += f", vs the true product {rt:.3f}"
        assert rt <= 1.0, msg
    print(msg)
    assert r <= 1.0, msg


def _lib():
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    L.load()
    L.init_device(torch.device("cuda"))
    return L


def st():
    return torch.cuda.current_stream().cuda_stream


def params(g, n, K):
    """Per-agent [W | b | gamma | beta | NaN pad]: W = w1t [K][256] (first layer) or natural [256 out][K in]."""
    ps = K * HID + 3 * HID + PAD
    P = torch.full((n, ps), float("nan"), device="cuda")
    P[:, :K * HID] = torch.randn(n, K * HID, device="cuda", generator=g) / math.sqrt(K)
    P[:, K * HID:K * HID + HID] = 0.1 * torch.randn(n, HID, device="cuda", generator=g)
    P[:, K * HID + HID:K * HID + 2 * HID] = 1.0 + 0.2 * torch.randn(n, HID, device="cuda", generator=g)
    P[:, K * HID + 2 * HID:K * HID + 3 * HID] = 0.2 * torch.randn(n, HID, device="cuda", generator=g)
    vec = lambda i: P[:, K * HID + i * HID:K * HID + (i + 1) * HID]
    return P, ps, vec


def stack(L, n, ps, lo=0, ctr=0):
    return L.Stack(n, 0, ps, lo, 0, ctr, 0, None) if n > 1 else None


def byref(s):
    return None if s is None else C.byref(s)


# ---- b2rl_tc_split_lo --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_agents,n", [(1, 1), (1, 3), (1, 4), (1, 7), (1, 65537), (3, 1022), (5, 65536)])
def test_tc_split_lo_bitwise(n_agents, n):
    """lo = x - hi(x) bit for bit (numpy mask), the n % 4 tail (tc_linear.cu:819), stacked agents with param / lo strides."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(n + n_agents)
    ps, ls = n + 4 + (-n) % 4, n + 12 + (-n) % 4
    W = torch.full((n_agents, ps), float("nan"), device="cuda")
    W[:, :n] = torch.randn(n_agents, n, device="cuda", generator=g) * torch.exp(4 * torch.randn(n_agents, n, device="cuda", generator=g))
    lo_f, lo = guarded(n_agents, ls)
    stk = L.Stack(n_agents, 0, ps, ls, 0, 0, 0, None) if n_agents > 1 else None
    L.check(L.load().b2rl_tc_split_lo(W.data_ptr(), lo.data_ptr(), n, byref(stk), st()), "tc_split_lo")
    torch.cuda.synchronize()
    w = W[:, :n].cpu().numpy()
    want = w - (w.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    assert np.array_equal(lo[:, :n].cpu().numpy().view(np.uint32), want.view(np.uint32))
    m = torch.zeros_like(lo, dtype=torch.bool)
    m[:, n:] = True
    untouched(lo_f, lo, m, "tc_split_lo")


# ---- b2rl_tc_linear (and b2rl_tc_linear_q's H / XH / stat) -------------------------------------------------------------------
def run_linear(L, X, M, n, P, ps, vec, prec, ln, relu, want_xh=True, want_stat=True):
    """One b2rl_tc_linear launch into guarded outputs; PREC 1 gets its lo mirror from b2rl_tc_split_lo."""
    lib = L.load()
    lo_buf, ls = None, 0
    if prec == "x3w":
        ls = HID * HID + PAD
        lo_buf = torch.full((n, ls), float("nan"), device="cuda")
        L.check(lib.b2rl_tc_split_lo(P.data_ptr(), lo_buf.data_ptr(), HID * HID, byref(L.Stack(n, 0, ps, ls, 0, 0, 0, None)), st()),
                "split")
    stk = stack(L, n, ps, ls)
    H_f, H = guarded(n * M, HID)
    XH_f, XH = guarded(n * M, HID)
    S_f, S = guarded(n * M, 2)
    wlo = {"tf32": None, "x3w": None if lo_buf is None else lo_buf.data_ptr(), "x3": P.data_ptr()}[prec]
    L.check(lib.b2rl_tc_linear(X.data_ptr(), HID, M, P.data_ptr(), wlo, vec(0).data_ptr(), vec(1).data_ptr() if ln else None,
                               vec(2).data_ptr() if ln else None, ln, relu, H.data_ptr(), XH.data_ptr() if want_xh else None,
                               S.data_ptr() if want_stat else None, byref(stk), st()), "tc_linear")
    return dict(H=H, H_f=H_f, XH=XH, XH_f=XH_f, S=S, S_f=S_f)


def check_forward(kernel, tag, acc, true, sabs, vec, n, M, prec, ln, relu, epw8, o, want_xh=True, want_stat=True):
    v = lambda i: vec(i).double()
    stat = o["S"].view(n, M, 2) if (ln and want_stat) else None
    xh = o["XH"].view(n, M, HID) if want_xh else None
    ref = fwd_ref(acc, v(0), v(1), v(2), ln, relu, epw8, stat, xh)
    if ln and want_stat:
        check(kernel, f"mean: {tag}", stat[..., 0], ref["mean"])
        check(kernel, f"rstd: {tag}", stat[..., 1], ref["rstd"])
    if want_xh:
        tr = None
        if not ln:  # the pre-activation IS the product (+ bias): the looser check against the true product
            z = true + v(0)[:, None, :]
            tr = (z, acc.e + T_TRUE[prec] * sabs + U * z.abs() + U * (acc.v + v(0)[:, None, :]).abs())
        check(kernel, f"x-hat: {tag}" if ln else f"pre-activation: {tag}", xh, ref["xh"], tr)
    check(kernel, f"H: {tag}", o["H"].view(n, M, HID), ref["h"])
    untouched(o["H_f"], what=f"{kernel} H")
    untouched(o["XH_f"], o["XH"], None if want_xh else torch.ones_like(o["XH"], dtype=torch.bool), f"{kernel} XH")
    untouched(o["S_f"], o["S"], None if (ln and want_stat) else torch.ones_like(o["S"], dtype=torch.bool), f"{kernel} stat")


FWD_CASES = [  # n agents, rows per agent, precision, LayerNorm, ReLU, x-hat stored, stat stored
    (1, 1, "tf32", 1, 1, 1, 1), (1, 32, "x3w", 1, 1, 1, 1), (1, 127, "x3", 1, 1, 1, 1), (1, 128, "tf32", 0, 1, 1, 1),
    (1, 129, "x3w", 0, 0, 1, 1), (1, 200, "x3", 1, 0, 0, 1), (1, 257, "tf32", 1, 1, 1, 0), (1, 1000, "x3w", 1, 1, 0, 0),
    (1, 65536, "tf32", 1, 1, 1, 1), (1, 65536, "x3w", 1, 1, 1, 1), (1, 65536, "x3", 0, 1, 1, 1),
    (160, 256, "x3", 1, 1, 1, 1), (160, 256, "tf32", 1, 1, 1, 1), (300, 200, "x3", 1, 1, 1, 1), (3, 1000, "x3w", 1, 1, 1, 1),
    (2, 40000, "x3", 1, 1, 1, 1), (2, 40000, "tf32", 0, 1, 1, 1), (1024, 256, "x3", 1, 1, 1, 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,prec,ln,relu,wx,ws", FWD_CASES)
def test_tc_linear_matches_float64(n, M, prec, ln, relu, wx, ws):
    """PREC 0 / 1 / 2, LayerNorm and ReLU on / off, x-hat and stat stored or not; M across the 128-row tile and the pair;
    stacked launches of more than 74 pairs (160 x 256, 300 x 200, 1 024 x 256: clusters change agent between tiles and
    swap vector sets) and 2 x 40 000 (a cluster's consecutive pairs sometimes of the same agent)."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(7 * M + n + len(prec))
    P, ps, vec = params(g, n, HID)
    X = torch.randn(n * M, HID, device="cuda", generator=g)
    o = run_linear(L, X, M, n, P, ps, vec, prec, ln, relu, bool(wx), bool(ws))
    torch.cuda.synchronize()
    acc, true, sabs = mma_acc(X.view(n, M, HID), P[:, :HID * HID].view(n, HID, HID), prec)
    check_forward("tc_linear", f"{prec} n={n} M={M} ln={ln} relu={relu}", acc, true, sabs, vec, n, M, prec, ln, relu,
                  prec == "tf32", o, bool(wx), bool(ws))


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,prec", [(1, 1000, "x3"), (3, 200, "x3"), (1, 300, "tf32")])
def test_tc_linear_q_hidden_layer_equals_tc_linear(n, M, prec):
    """b2rl_tc_linear_q runs the same kernel with the critic head in its epilogue: its H / XH / stat equal b2rl_tc_linear's
    bit for bit on the same inputs."""
    L = _lib()
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(M + n)
    P, ps, vec = params(g, n, HID)
    X = torch.randn(n * M, HID, device="cuda", generator=g)
    o = run_linear(L, X, M, n, P, ps, vec, prec, 1, 1)
    w3 = torch.randn(n, ps, device="cuda", generator=g) / 16.0
    q = L.WideQ()
    qo = torch.empty(n * M, device="cuda")
    q.h2, q.w3, q.b3, q.q_out, q.M, q.mode = None, w3.data_ptr(), w3.data_ptr() + 4 * HID, qo.data_ptr(), M, 0
    H, XH, S = torch.empty(n * M, HID, device="cuda"), torch.empty(n * M, HID, device="cuda"), torch.empty(n * M, 2, device="cuda")
    L.check(lib.b2rl_tc_linear_q(X.data_ptr(), HID, M, P.data_ptr(), P.data_ptr() if prec == "x3" else None, vec(0).data_ptr(),
                                 vec(1).data_ptr(), vec(2).data_ptr(), 1, H.data_ptr(), XH.data_ptr(), S.data_ptr(), C.byref(q),
                                 byref(stack(L, n, ps)), st()), "tc_linear_q")
    torch.cuda.synchronize()
    assert torch.equal(H, o["H"]) and torch.equal(XH, o["XH"]) and torch.equal(S, o["S"])


# ---- b2rl_tc_first and b2rl_wide_first ------------------------------------------------------------------------------------
def first_inputs(g, n, M, K):
    ldx = K + 4 - K % 4 if K % 4 else K + 4  # (ldx > K, a multiple of 4: the columns between are NaN)
    X = torch.full((n * M, ldx), float("nan"), device="cuda")
    X[:, :K] = torch.randn(n * M, K, device="cuda", generator=g)
    return X, ldx


FIRST_CASES = [(1, M, K) for M, K in zip((1, 32, 127, 128, 129, 200, 257, 1000, 65536, 300),
                                         (1, 5, 11, 14, 27, 32, 33, 35, 376, 393))] + [
    (160, 256, 14), (300, 200, 27), (2, 40000, 35), (1024, 256, 17)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,K", FIRST_CASES)
def test_first_layers_match_float64(n, M, K):
    """tc_first in TF32 and 3xTF32 (one / two / twelve / thirteen k-slabs, ldx > K with NaN between) and the FFMA
    wide_first on the same inputs; stacked launches of more than 74 pairs and 2 x 40 000."""
    L = _lib()
    lib = L.load()
    g = torch.Generator(device="cuda").manual_seed(M + K + n)
    P, ps, vec = params(g, n, K)
    X, ldx = first_inputs(g, n, M, K)
    stk = stack(L, n, ps)
    ln = 0 if K == 33 else 1  # (one case without LayerNorm: the pre-activation is the product)
    outs = {}
    for fn in ("tf32", "x3", "ffma"):
        o = dict(zip(("H_f", "H", "XH_f", "XH", "S_f", "S"), (*guarded(n * M, HID), *guarded(n * M, HID), *guarded(n * M, 2))))
        args = (X.data_ptr(), ldx, M, K, P.data_ptr(), vec(0).data_ptr(), vec(1).data_ptr(), vec(2).data_ptr(), ln, o["H"].data_ptr(),
                o["XH"].data_ptr(), o["S"].data_ptr())
        if fn == "ffma":
            L.check(lib.b2rl_wide_first(*args, byref(stk), st()), "wide_first")
        else:
            L.check(lib.b2rl_tc_first(*args, int(fn == "x3"), byref(stk), st()), "tc_first")
        outs[fn] = o
    torch.cuda.synchronize()
    Xk = X[:, :K].reshape(n, M, K)
    W = P[:, :K * HID].view(n, K, HID).mT
    for prec in ("tf32", "x3"):
        acc, true, sabs = mma_acc(Xk, W, prec)
        check_forward("tc_first", f"{prec} n={n} M={M} K={K}", acc, true, sabs, vec, n, M, prec, ln, 1, True, outs[prec])
    # FFMA: the sequential chain over K (wide.cu:53-86), then the two-pass LayerNorm of wide.cu:104-118
    o = outs["ffma"]
    Xd, Wd = Xk.double(), W.double()
    z = R(Xd @ Wd.mT, gam(K) * (Xd.abs() @ Wd.abs().mT)) + R(vec(0).double()[:, None, :])
    tag = f"n={n} M={M} K={K}"
    if ln:
        mean = r_sum(z, -1, 8) * (1.0 / HID)
        d = z - R(mean.v[..., None], mean.e[..., None])
        rstd = R(1.0) / r_sqrt(r_sum(d * d, -1, 13) * (1.0 / HID) + LN_EPS)
        S = o["S"].view(n, M, 2)
        check("wide_first", f"mean: {tag}", S[..., 0], mean)
        check("wide_first", f"rstd: {tag}", S[..., 1], rstd)
        xh = (z - R(S[..., :1])) * R(S[..., 1:])
        check("wide_first", f"x-hat: {tag}", o["XH"].view(n, M, HID), xh)
        y = r_relu(R(o["XH"].view(n, M, HID)) * R(vec(1).double()[:, None, :]) + R(vec(2).double()[:, None, :]))
    else:
        untouched(o["S_f"], o["S"], torch.ones_like(o["S"], dtype=torch.bool), "wide_first stat")
        y = r_relu(z)
    check("wide_first", f"H: {tag}", o["H"].view(n, M, HID), y)
    untouched(o["H_f"], what="wide_first H")
    untouched(o["XH_f"], what="wide_first XH")


# ---- b2rl_tc_linear_bwd ---------------------------------------------------------------------------------------------------
def bwd_inputs(g, n, M):
    P, ps, vec = params(g, n, HID)  # [w2t | (unused) | gamma | beta | pad]
    DZ2 = torch.randn(n * M, HID, device="cuda", generator=g)
    XH = torch.randn(n * M, HID, device="cuda", generator=g)
    stat = torch.stack([torch.randn(n * M, device="cuda", generator=g), 0.5 + torch.rand(n * M, device="cuda", generator=g)], 1)
    return P, ps, vec, DZ2, XH, stat.contiguous()


def run_bwd(L, n, M, P, ps, vec, DZ2, XH, stat, prec, ln, with_part):
    lib = L.load()
    lo_buf, ls = None, 0
    if prec == "x3w":
        ls = HID * HID + PAD
        lo_buf = torch.full((n, ls), float("nan"), device="cuda")
        L.check(lib.b2rl_tc_split_lo(P.data_ptr(), lo_buf.data_ptr(), HID * HID, byref(L.Stack(n, 0, ps, ls, 0, 0, 0, None)), st()),
                "split")
    nt = (M + 127) // 128
    D_f, D = guarded(n * M, HID)
    p_f, part = guarded(n, nt, 3, HID)
    wlo = {"tf32": None, "x3w": None if lo_buf is None else lo_buf.data_ptr(), "x3": P.data_ptr()}[prec]
    L.check(lib.b2rl_tc_linear_bwd(DZ2.data_ptr(), M, P.data_ptr(), wlo, XH.data_ptr(), stat.data_ptr(),
                                   vec(1).data_ptr() if ln else None, vec(2).data_ptr() if ln else None, ln, D.data_ptr(),
                                   part.data_ptr() if with_part else None, byref(stack(L, n, ps, ls)), st()), "tc_linear_bwd")
    return D, D_f, part, p_f


def bwd_ref(dh: R, x, rstd, gm, be, ln):
    """dz1 and dn from dh = dz2 . W2 (R): the ReLU mask and the LayerNorm backward of tc_linear.cu:660-712."""
    on = (x * gm + be) > 0 if ln else x > 0  # (exact: fma rounds once and keeps the sign)
    dn = R(torch.where(on, dh.v, 0.0), torch.where(on, dh.e, 0.0))
    if not ln:
        return dn, dn
    X, G = R(x), R(gm.expand_as(x))
    dx = dn * G
    m1, m2 = r_sum(dx, -1, 128) * (1.0 / HID), r_sum(dx * X, -1, 128) * (1.0 / HID)
    dz = R(rstd[..., None]) * ((dx - R(m1.v[..., None], m1.e[..., None])) - X * R(m2.v[..., None], m2.e[..., None]))
    return dz, dn


def tile_sums(a: R, rows_per_tile, k):
    """[n, M, 256] -> [n, T, 256]: sums over consecutive tiles of rows (a ragged last tile padded with exact zeros)."""
    n, M = a.v.shape[:2]
    pad = (-M) % rows_per_tile
    f = lambda t: torch.cat([t, t.new_zeros(n, pad, t.shape[2])], 1).view(n, -1, rows_per_tile, t.shape[2])
    return r_sum(R(f(a.v), f(a.e)), 2, k)


BWD_CASES = [(1, 1, "tf32", 1, 1), (1, 32, "x3", 1, 1), (1, 127, "x3w", 1, 0), (1, 129, "tf32", 0, 1), (1, 200, "x3", 0, 1),
             (1, 1000, "x3w", 1, 1), (1, 65536, "tf32", 1, 1), (1, 65536, "x3", 1, 1), (160, 256, "x3", 1, 1),
             (300, 200, "tf32", 1, 1), (2, 40000, "x3", 1, 1), (1024, 256, "x3", 1, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,M,prec,ln,with_part", BWD_CASES)
def test_tc_linear_bwd_matches_float64(n, M, prec, ln, with_part):
    """dz1 and each tile's three column-sum partials separately: PREC 0 / 1 / 2, LayerNorm on / off, part NULL or given,
    ragged tiles, stacked launches of more than 74 pairs."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(11 * M + n + len(prec))
    P, ps, vec, DZ2, XH, stat = bwd_inputs(g, n, M)
    D, D_f, part, p_f = run_bwd(L, n, M, P, ps, vec, DZ2, XH, stat, prec, ln, with_part)
    torch.cuda.synchronize()
    dh, true, sabs = mma_acc(DZ2.view(n, M, HID), P[:, :HID * HID].view(n, HID, HID), prec)
    x = XH.view(n, M, HID).double()
    dz, dn = bwd_ref(dh, x, stat[:, 1].view(n, M).double(), vec(1).double()[:, None, :], vec(2).double()[:, None, :], ln)
    tag = f"{prec} n={n} M={M} ln={ln}"
    tr = None
    if not ln:
        on = x > 0
        tr = (torch.where(on, true, 0.0), torch.where(on, dh.e + T_TRUE[prec] * sabs, 0.0))
    check("tc_linear_bwd", f"dz1: {tag}", D.view(n, M, HID), dz, tr)
    untouched(D_f, what="tc_linear_bwd dz1")
    if with_part:
        pt = part.view(n, -1, 3, HID)
        check("tc_linear_bwd", f"partial sum dz: {tag}", pt[:, :, 0], tile_sums(R(D.view(n, M, HID)), 128, 33))
        check("tc_linear_bwd", f"partial sum dn x-hat: {tag}", pt[:, :, 1], tile_sums(R(x) * dn, 128, 33))
        check("tc_linear_bwd", f"partial sum dn: {tag}", pt[:, :, 2], tile_sums(dn, 128, 33))
        untouched(p_f, what="tc_linear_bwd part")
    else:
        untouched(p_f, part, torch.ones_like(part, dtype=torch.bool), "tc_linear_bwd part (NULL)")


# ---- b2rl_wide_ln_bwd -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,M,n_out,ln", [(1, 1, 1, 1), (1, 129, 6, 1), (1, 1000, 64, 1), (1, 1000, 1, 0), (1, 4097, 1, 1),
                                         (3, 200, 6, 1), (3, 257, 1, 1)])
def test_wide_ln_bwd_matches_float64(n, M, n_out, ln):
    """Head backward + ReLU mask + LayerNorm backward of layer 2, its per-CTA partials and the scalar head's dw3_part."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(M + n_out + n)
    ps = MAX_OUT * HID + 3 * HID + PAD  # [w3 | gamma | beta | ...]
    Pm = torch.full((n, ps), float("nan"), device="cuda")
    Pm[:, :n_out * HID] = torch.randn(n, n_out * HID, device="cuda", generator=g) / 16.0
    og = MAX_OUT * HID
    Pm[:, og:og + HID] = 1.0 + 0.2 * torch.randn(n, HID, device="cuda", generator=g)
    Pm[:, og + HID:og + 2 * HID] = 0.2 * torch.randn(n, HID, device="cuda", generator=g)
    dz3 = torch.full((n * M, MAX_OUT), float("nan"), device="cuda")
    dz3[:, :n_out] = torch.randn(n * M, n_out, device="cuda", generator=g)
    XH = torch.randn(n * M, HID, device="cuda", generator=g)
    stat = torch.stack([torch.randn(n * M, device="cuda", generator=g), 0.5 + torch.rand(n * M, device="cuda", generator=g)], 1).contiguous()
    nb = (M + 127) // 128
    D_f, D = guarded(n * M, HID)
    p_f, part = guarded(n, nb, 3, HID)
    w_f, dw3 = guarded(n, nb, 3, HID)
    L.check(L.load().b2rl_wide_ln_bwd(dz3.data_ptr(), n_out, Pm.data_ptr(), XH.data_ptr(), stat.data_ptr(), Pm.data_ptr() + 4 * og,
                                      Pm.data_ptr() + 4 * (og + HID), ln, M, D.data_ptr(), part.data_ptr(),
                                      dw3.data_ptr() if n_out == 1 else None, byref(stack(L, n, ps)), st()), "wide_ln_bwd")
    torch.cuda.synchronize()
    d = dz3[:, :n_out].view(n, M, n_out).double()
    w3 = Pm[:, :n_out * HID].view(n, n_out, HID).double()
    dh = R(d @ w3, gam(n_out) * (d.abs() @ w3.abs()))
    x = XH.view(n, M, HID).double()
    gm, be = Pm[:, og:og + HID].double()[:, None, :], Pm[:, og + HID:og + 2 * HID].double()[:, None, :]
    on = (x * gm + be) > 0 if ln else x > 0
    dn = R(torch.where(on, dh.v, 0.0), torch.where(on, dh.e, 0.0))
    if ln:
        X, G = R(x), R(gm.expand_as(x))
        dx = dn * G
        m1, m2 = r_sum(dx, -1, 13) * (1.0 / HID), r_sum(dx * X, -1, 13) * (1.0 / HID)
        dz = R(stat[:, 1].view(n, M, 1).double()) * ((dx - R(m1.v[..., None], m1.e[..., None])) - X * R(m2.v[..., None], m2.e[..., None]))
    else:
        dz = dn
    tag = f"n={n} M={M} n_out={n_out} ln={ln}"
    check("wide_ln_bwd", f"dz2: {tag}", D.view(n, M, HID), dz)
    pt = part.view(n, nb, 3, HID)
    check("wide_ln_bwd", f"partial sum dz: {tag}", pt[:, :, 0], tile_sums(R(D.view(n, M, HID)), 128, 24))
    check("wide_ln_bwd", f"partial sum dn x-hat: {tag}", pt[:, :, 1], tile_sums(R(x) * dn, 128, 24))
    check("wide_ln_bwd", f"partial sum dn: {tag}", pt[:, :, 2], tile_sums(dn, 128, 24))
    untouched(D_f, what="wide_ln_bwd dz")
    untouched(p_f, what="wide_ln_bwd part")
    if n_out == 1:
        pre = R(x * gm + be, U * (x * gm + be).abs()) if ln else R(x)
        hr = R(torch.where(on, pre.v, 0.0), torch.where(on, pre.e, 0.0))
        check("wide_ln_bwd", f"dw3 partial: {tag}", dw3.view(n, nb, 3, HID)[:, :, 0], tile_sums(R(d) * hr, 128, 24))
        m = torch.zeros_like(dw3, dtype=torch.bool)
        m[:, :, 1:] = True
        untouched(w_f, dw3, m, "wide_ln_bwd dw3_part (slots 1, 2)")
    else:
        untouched(w_f, dw3, torch.ones_like(dw3, dtype=torch.bool), "wide_ln_bwd dw3_part (NULL)")


# ---- b2rl_tc_wgrad ---------------------------------------------------------------------------------------------------------
def wgrad_splits(Bn, MA, stacked):  # tc_wgrad.cu tc_wgrad_splits
    mt = (MA + 127) // 128
    cap = (148 + mt - 1) // mt
    s = (Bn + 1023) // 1024 if stacked else (Bn + 127) // 128
    return max(1, min(s, cap))


def wgrad_ref(A, Bm, prec, S):
    """A [n, Bn, MA], Bm [n, Bn, 256] -> (per-split slices R [n, S, MA, 256], the reduce's C R [n, MA, 256], true, sum|ab|)."""
    n, Bn, MA = A.shape
    rps = ((Bn + S - 1) // S + 31) // 32 * 32
    pad = S * rps - Bn
    f = lambda t: torch.cat([t, t.new_zeros(n, pad, t.shape[2])], 1).view(n, S, rps, t.shape[2]).mT
    sl, _, _ = mma_acc(f(A), f(Bm), prec)
    red = None
    for w in range(8):  # tc_wgrad_reduce_kernel: warp w adds slices w, w + 8, ...; then the warps in order
        idx = list(range(w, S, 8))
        if not idx:
            continue
        a = sl[:, idx[0]]
        for s in idx[1:]:
            a = a + sl[:, s]
        red = a if red is None else red + a
    Ad, Bd = A.double(), Bm.double()
    return sl, red, Ad.mT @ Bd, Ad.abs().mT @ Bd.abs()


def run_wgrad(L, A, lda, MA, Bm, Bn, n, x3, transpose, bump_base=7):
    """One launch into guarded gradient tensors (stacked: param_stride apart with NaN between) and NaN scratch."""
    lib = L.load()
    ps = (2 if transpose else 1) * (MA * HID + PAD)
    G_f, G = guarded(n, ps)
    ctr = torch.full((n, 8), bump_base, dtype=torch.int64, device="cuda")
    scratch = torch.full((lib.b2rl_tc_wgrad_scratch_floats(MA, Bn, n if n > 1 else 0),), float("nan"), device="cuda")
    stk = L.Stack(n, 0, ps, 0, 0, 8, 0, None) if n > 1 else None
    Ct = G.data_ptr() + 4 * (MA * HID + PAD) if transpose else None
    L.check(lib.b2rl_tc_wgrad(A.data_ptr(), lda, lda, MA, Bm.data_ptr(), Bn, G.data_ptr(), Ct, scratch.data_ptr(), int(x3),
                              ctr.data_ptr() + 8, byref(stk), st()), "tc_wgrad")
    return G, G_f, ctr


WGRAD_GRID = [(Bn, MA, x3) for Bn in (1, 31, 32, 33, 1000, 4097) for MA in (1, 6, 11, 17, 64, 128, 129, 256, 376, 393)
              for x3 in (0, 1)]
WGRAD_CASES = ([(1, Bn, MA, x3) for Bn, MA, x3 in WGRAD_GRID]
               + [(1, 65536, MA, x3) for MA in (1, 6, 64, 128, 129, 256, 393) for x3 in (0, 1)]
               + [(1024, 256, 256, 1), (1024, 256, 256, 0), (1024, 256, 11, 1), (1024, 256, 11, 0), (300, 2500, 256, 1),
                  (300, 2500, 11, 0), (3, 1000, 393, 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("n,Bn,MA,x3", WGRAD_CASES)
def test_tc_wgrad_matches_float64(n, Bn, MA, x3):
    """C = A^T B per agent: TF32, 3xTF32 single-SM and PAIR (129..256 rows); Bn across the 32-row slab and the splits,
    65 536 with MA <= 128 (the last split empty), stacked 1 024 x 256 (the direct path, many items per CTA) and 300 x 2 500
    (three splits: the reduce path over 300 agents); Ct bitwise the transpose; each agent's counter advanced by one."""
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(Bn + 3 * MA + n + x3)
    lda = MA + 4 - MA % 4 + 4
    A = torch.full((n * Bn, lda), float("nan"), device="cuda")
    A[:, :MA] = torch.randn(n * Bn, MA, device="cuda", generator=g)  # (columns MA.. are NaN: rows the kernel must not store)
    Bm = torch.randn(n * Bn, HID, device="cuda", generator=g)
    transpose = MA % 4 == 0
    G, G_f, ctr = run_wgrad(L, A, lda, MA, Bm, Bn, n, x3, transpose)
    torch.cuda.synchronize()
    S = wgrad_splits(Bn, MA, n > 1)
    prec = "x3" if x3 else "tf32"
    sl, red, true, sabs = wgrad_ref(A[:, :MA].reshape(n, Bn, MA), Bm.view(n, Bn, HID), prec, S)
    ref = sl[:, 0] if (n > 1 and S == 1) else red
    Cg = G[:, :MA * HID].view(n, MA, HID)
    path = ("PAIR" if (x3 and (MA + 127) // 128 == 2) else "single-SM") + (", direct" if n > 1 and S == 1 else f", S={S}")
    check("tc_wgrad", f"{prec} C: n={n} Bn={Bn} MA={MA} ({path})", Cg, ref, (true, ref.e + T_TRUE[prec] * sabs))
    owned = torch.zeros_like(G, dtype=torch.bool)
    owned[:, :MA * HID] = True
    if transpose:
        o = MA * HID + PAD
        assert torch.equal(G[:, o:o + MA * HID].view(n, HID, MA), Cg.mT), "Ct is not the transpose of C"
        owned[:, o:o + MA * HID] = True
    untouched(G_f, G, ~owned, "tc_wgrad C / Ct")
    want = torch.full_like(ctr, 7)
    want[:, 1] = 8
    assert torch.equal(ctr, want), "bump: one per agent, in slot 1 only"


# ---- stacked contract at scale: sharding and repeated launches ----------------------------------------------------------------
@pytest.mark.gpu
def test_stacked_launches_are_shard_invariant_and_reproducible():
    """1 024 agents x 256 rows (BASELINE config 4): one launch of each entry point equals, bit for bit, two launches over the
    shards [0, 600) and [600, 1 024) (DESIGN §3.5b), and three launches of the stacked PREC-2 forward and backward and of the
    stacked PAIR weight gradient agree bitwise (the stacked form of test_tc_kernels_are_reproducible_at_full_grid)."""
    L = _lib()
    lib = L.load()
    n, M, cut, K = 1024, 256, 600, 17
    g = torch.Generator(device="cuda").manual_seed(1024)
    P, ps, vec = params(g, n, HID)
    P1, ps1, vec1 = params(g, n, K)
    X = torch.randn(n * M, HID, device="cuda", generator=g)
    X1, ldx = first_inputs(g, n, M, K)
    DZ2 = torch.randn(n * M, HID, device="cuda", generator=g)
    stat0 = torch.stack([torch.zeros(n * M, device="cuda"), 0.5 + torch.rand(n * M, device="cuda", generator=g)], 1).contiguous()
    nt = (M + 127) // 128

    def launches(a0, a1):
        """Every entry point over agents [a0, a1): outputs of the shard."""
        m = a1 - a0
        stk = lambda s: C.byref(L.Stack(m, a0, s, 0, 0, 8, 0, None))
        o = {k: torch.full((m * M, HID), float("nan"), device="cuda") for k in ("H", "XH", "H1", "XH1", "DZ1")}
        o["S"], o["S1"] = (torch.full((m * M, 2), float("nan"), device="cuda") for _ in range(2))
        o["part"] = torch.full((m, nt, 3, HID), float("nan"), device="cuda")
        p, p1 = P.data_ptr() + 4 * a0 * ps, P1.data_ptr() + 4 * a0 * ps1
        vp = lambda v, i: v(i).data_ptr() + 4 * a0 * (ps if v is vec else ps1)
        L.check(lib.b2rl_tc_linear(X.data_ptr() + 4 * a0 * M * HID, HID, M, p, p, vp(vec, 0), vp(vec, 1), vp(vec, 2), 1, 1,
                                   o["H"].data_ptr(), o["XH"].data_ptr(), o["S"].data_ptr(), stk(ps), st()), "tc_linear")
        L.check(lib.b2rl_tc_first(X1.data_ptr() + 4 * a0 * M * ldx, ldx, M, K, p1, vp(vec1, 0), vp(vec1, 1), vp(vec1, 2), 1,
                                  o["H1"].data_ptr(), o["XH1"].data_ptr(), o["S1"].data_ptr(), 1, stk(ps1), st()), "tc_first")
        L.check(lib.b2rl_tc_linear_bwd(DZ2.data_ptr() + 4 * a0 * M * HID, M, p, p, X.data_ptr() + 4 * a0 * M * HID,
                                       stat0.data_ptr() + 8 * a0 * M, vp(vec, 1), vp(vec, 2), 1, o["DZ1"].data_ptr(),
                                       o["part"].data_ptr(), stk(ps), st()), "tc_linear_bwd")
        for MA, x3 in ((256, 1), (11, 0)):
            wps = 2 * MA * HID + 8
            Gw = torch.full((m, wps), float("nan"), device="cuda")
            ctr = torch.zeros(m, 8, dtype=torch.int64, device="cuda")
            scr = torch.full((lib.b2rl_tc_wgrad_scratch_floats(MA, M, m),), float("nan"), device="cuda")
            L.check(lib.b2rl_tc_wgrad(o["H"].data_ptr(), HID, HID, MA, o["DZ1"].data_ptr(), M, Gw.data_ptr(),
                                      Gw.data_ptr() + 4 * (MA * HID + 4) if MA % 4 == 0 else None, scr.data_ptr(), x3,
                                      ctr.data_ptr(), stk(wps), st()), "tc_wgrad")
            o[f"G{MA}"], o[f"ctr{MA}"] = Gw, ctr
        torch.cuda.synchronize()
        return o

    same = lambda a, b: torch.equal(a.view(torch.int32), b.view(torch.int32)) if a.is_floating_point() else torch.equal(a, b)
    full = launches(0, n)
    for k, t in full.items():
        assert not t.is_floating_point() or torch.isfinite(t if k[0] != "G" else t[:, :int(k[1:]) * HID]).all(), k
    lo, hi_ = launches(0, cut), launches(cut, n)
    for k in full:
        assert same(full[k], torch.cat([lo[k], hi_[k]])), f"{k}: the sharded launches differ from the whole population's"
    for it in range(2):
        again = launches(0, n)
        for k in ("H", "XH", "S", "DZ1", "part", "G256"):
            assert same(full[k], again[k]), f"launch {it + 2}: {k} differs from the first launch"


@pytest.mark.gpu
def test_report_worst_ratios():
    """(runs last in this module) the worst deviation / bound ratio of each kernel and output over the tests above."""
    for k, v in sorted(WORST.items()):
        print(f"worst dev/bound {k:40s} {v:.3f}")


# ---- the bounds have teeth (no GPU) --------------------------------------------------------------------------------------
def _teeth(name, wrong, ref: R, at_least=10.0):
    ratio = float(((wrong.double() - ref.v).abs() / (WIDEN * ref.e + FLOOR)).max())
    print(f"{name}: {ratio:.1f} x the bound")
    assert ratio >= at_least, f"{name}: the bound accepts this mistake (worst ratio {ratio:.2f})"
    return ratio


def test_bounds_have_teeth():
    """On the CPU, at small shapes: each bound rejects, at least tenfold, a mistake applied to the float64 reference —
    another agent's bias / gamma / beta for one tile, a tile row from the neighbouring agent, one k-slab dropped, 3xTF32
    without either lo product, a split slice dropped or counted twice, a tile's partial in its neighbour's slot, rstd from
    the neighbouring row. One lo product dropped on a single k-slab (8 products of 2^-11 relative size among 768) is
    near the accumulation bound at K = 256; its factor is reported, not required."""
    g = torch.Generator().manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g)
    n, M = 2, 256
    X = rn(n, M, HID)
    W = rn(n, HID, HID) / 16.0
    b, gm, be = 0.1 * rn(n, HID), 1.0 + 0.2 * rn(n, HID), 0.2 * rn(n, HID)
    for prec in ("tf32", "x3"):
        acc, _, _ = mma_acc(X, W, prec)
        ref = fwd_ref(acc, b.double(), gm.double(), be.double(), 1, 1, prec == "tf32")
        for name, (b2, g2, be2) in {"bias": (b.flip(0), gm, be), "gamma": (b, gm.flip(0), be), "beta": (b, gm, be.flip(0))}.items():
            wr = fwd_ref(acc, b2.double(), g2.double(), be2.double(), 1, 1, prec == "tf32")["h"].v
            wrong = ref["h"].v.clone()
            wrong[0, :128] = wr[0, :128]  # one tile of agent 0 with agent 1's vector
            _teeth(f"{prec} H, another agent's {name} for one tile", wrong, ref["h"])
        wrong = ref["h"].v.clone()
        acc1, _, _ = mma_acc(X.flip(0), W, prec)
        wrong[0, 5] = fwd_ref(acc1, b.double(), gm.double(), be.double(), 1, 1, prec == "tf32")["h"].v[0, 5]
        _teeth(f"{prec} H, a tile row from the neighbouring agent", wrong, ref["h"])
        xs = lambda k0, k1, f: f(X[..., k0:k1]).double() @ f(W[..., k0:k1]).double().mT
        _teeth(f"{prec} pre-activation, one k-slab dropped", acc.v - xs(64, 96, hi), acc)
        rs = ref["rstd"].v
        _teeth(f"{prec} x-hat, rstd from the neighbouring row", (acc.v + b.double()[:, None] - ref["mean"].v[..., None]) *
               rs.roll(1, 1)[..., None], ref["xh"])
    acc, _, _ = mma_acc(X, W, "x3")
    _teeth("3xTF32, no lo(a).hi(b)", acc.v - lo3(X).double() @ hi(W).double().mT, acc)
    _teeth("3xTF32, no hi(a).lo(b)", acc.v - hi(X).double() @ lo3(W).double().mT, acc)
    one = float(((hi(X[..., 64:72]).double() @ lo3(W[..., 64:72]).double().mT).abs() / (WIDEN * acc.e + FLOOR)).max())
    one_slab = float(((hi(X[..., 64:96]).double() @ lo3(W[..., 64:96]).double().mT).abs() / (WIDEN * acc.e + FLOOR)).max())
    print(f"3xTF32, one hi.lo' instruction dropped: {one:.1f} x the bound; one k-slab's hi.lo' products: {one_slab:.1f} x")
    # tc_linear_bwd: a tile's partial in its neighbour's slot, rstd from the neighbouring row
    DZ2, XH = rn(n, M, HID), rn(n, M, HID)
    rstd = 0.5 + torch.rand(n, M, generator=g)
    dh, _, _ = mma_acc(DZ2, W, "x3")
    args = (XH.double(), None, gm.double()[:, None], be.double()[:, None], 1)
    dz, dn = bwd_ref(dh, args[0], rstd.double(), *args[2:])
    wz, _ = bwd_ref(dh, args[0], rstd.roll(1, 1).double(), *args[2:])
    _teeth("dz1, rstd from the neighbouring row", wz.v, dz)
    p = tile_sums(dn, 128, 33)
    _teeth("partial sum dn, written to the neighbour's tile slot", p.v.flip(1), p)
    p = tile_sums(R(XH.double()) * dn, 128, 33)
    _teeth("partial sum dn x-hat, written to the neighbour's tile slot", p.v.flip(1), p)
    # tc_wgrad: a split slice dropped or counted twice
    A, Bm = rn(1, 1000, 64), rn(1, 1000, HID)
    S = wgrad_splits(1000, 64, False)
    sl, red, _, _ = wgrad_ref(A, Bm, "x3", S)
    _teeth("tc_wgrad, a split slice dropped", red.v - sl.v[:, 3], red)
    _teeth("tc_wgrad, a split slice counted twice", red.v + sl.v[:, 3], red)
    acc, _, _ = mma_acc(A.mT, Bm.mT, "tf32")
    _teeth("tc_wgrad TF32, one 32-row slab dropped", acc.v - hi(A[:, 32:64]).double().mT @ hi(Bm[:, 32:64]).double(),
           wgrad_ref(A, Bm, "tf32", S)[1])
