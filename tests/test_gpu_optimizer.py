"""The optimizer kernels against a float64 restatement of Adam, element by element.

Every parameter of every learner goes through one of three optimizers: adam_polyak_multi (csrc/adam.cu), the Adam fused
into the weight-gradient kernel (b2rl_*_update_opt, csrc/wgrad.cu; both use csrc/adam_math.cuh) and the scalar Adam of
the temperature step (csrc/actor.cu, adam_scalar). The reference below is torch's `capturable` branch in float64:

    g  = g * gscale                                 gscale = grad_scale * min(1, clip / (||g * grad_scale|| + 1e-6))
    m' = m + (1 - b1)(g - m)                        v' = b2 v + (1 - b2) g^2
    ss = -lr / (1 - b1^t)                           denom = sqrt(v') / (sqrt(1 - b2^t) ss) + eps / ss
    p' = p + m' / denom                             T' = T + tau (p' - T)   (Polyak, with the NEW p)

It takes the hyperparameters as the fp32 values the kernel receives (np.float32(0.999) widened to float64: the kernel's
1 - beta is then exact by Sterbenz, so the constants agree), t as the exact integer, and it runs one step from the
pre-step state read back from the device: the bound is on the LOCAL error of one step, not on a drift.

Error bound of one step, per element (u = 2^-24, the unit roundoff of fp32; first order, then widened by 0.1 %):
  - gradient: eps_g = 0 when gscale is exactly 1, u for fl(g * grad_scale), and eps_c + 2u with clipping, where the
    clip coefficient's relative error eps_c = eps_ss / 2 + 4u follows from the sumsq bound below (sqrt halves it, then
    the product with grad_scale, the + 1e-6 and the division round once each).
  - m': fl(g - m) and the fma round once each:  E_m = (1 - b1) |g| eps_g + (1 - b1) |g - m| u + |m'| u.
    (adam_scalar of the temperature step may round the product (1 - b1)(g - m) as well: one more u on that term.)
  - v': its terms are non-negative: fl((1 - b2) g), fl(b2 v) and the fma give E_v = (1 - b2) g^2 2 eps_g + 2u v'
    (3u v' for adam_scalar, whose products may be rounded separately).
  - bias corrections: powf is within 4 ulp (CUDA C++ Programming Guide, "Mathematical Functions", single-precision
    table: powf(x, y), maximum ulp error 4, full range), i.e. 8u beta^t relative plus 4 * 2^-149 absolute where beta^t
    underflows; the kernel takes t as fl32(t), which moves beta^t by |ln beta| |t - fl32(t)| beta^t (t > 2^24). Then
    1 - beta^t rounds once: eps_bc = (8u beta^t + ...) / (1 - beta^t) + u. This is ill-conditioned at small t: the factor
    beta^t / (1 - beta^t) is 999.5 for b2 at t = 1, so eps_bc2 ~ 8000u there, and the bound on p' is mostly this term.
  - scalars: ssn = -(lr / bc1): eps_bc1 + u;  c1 = sqrt(bc2) ssn: eps_bc2 / 2 + u + eps_ssn + u;  c2 = eps / ssn: eps_ssn + u.
  - denom = fl(fl(sqrt(v') / c1) + c2): both terms have one sign, so eps_den = max(E_v / 2v' + 2u + eps_c1, eps_c2) + u.
  - p' = fl(p + fl(m' / denom)): E_p = E_m / |denom| + |m' / denom| (eps_den + u) + |p'| u.
  - Polyak: fl(p' - T) then the fma: E_T = tau E_p + tau |p' - T| u (1 + u) + |T'| u.
  - sumsq (b2rl_grad_sumsq), non-negative terms, so the relative error is the depth of the reduction times u:
    k fmas per thread (k = ceil(len / (64 * 256)), the grid stride), 5 shuffle levels, 8 warps and 64 per-CTA parts:
    eps_ss = (k + 77) u.
  - temperature: out[ALPHA] = expf(log_alpha'), expf within 2 ulp: 4u relative, + u for the stored log_alpha.
An absolute floor of 2^-140 covers subnormal results. The worst deviation / bound ratio of each group is printed. Ratios
close to 1 are expected of a correct kernel: the last rounding of p', m', v' or T' alone reaches u |x| where x lies just
above a power of two and the other terms are small, so the bound is tight there.
test_bound_has_teeth shows on the tests' own data that a fp32 emulation of the kernels stays inside the bound while each
of seven plausible mistakes exceeds it at least tenfold somewhere.
"""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from sac_td3_cudagraphs_pytorch_b200 import _lib as L
from sac_td3_cudagraphs_pytorch_b200.arena import make_layout, set_shadow_pairs

U = 2.0 ** -24
POW_ULP = 4      # powf, CUDA C++ Programming Guide, single-precision mathematical functions
EXP_ULP = 2      # expf, same table
FLOOR = 2.0 ** -140
WIDEN = 1.001    # (second-order terms)
f32 = lambda x: float(np.float32(x))
B1, B2, EPS, CLIP_EPS = f32(0.9), f32(0.999), f32(1e-8), f32(1e-6)
TAU = f32(0.005)
HH = L.HID * L.HID
TS = (1, 2, 3, 10, 1000, 2 ** 24 + 1, 2 ** 40)  # one stacked agent per step count
SENT = np.uint32(0x5EED5EED).view(np.float32)    # everything a launch must not write
QNAN = np.uint32(0x7FC0BEEF).view(np.float32)    # the shadows' own gradient / moments: never read


# ------------------------------------------------------------------------------------------------ the reference
def adam_ref(p, g, m, v, t, lr, b1=B1, b2=B2, eps=EPS):
    """One Adam step in float64 (g already scaled). t: exact step count(s), broadcast against the arrays."""
    m1 = m + (1.0 - b1) * (g - m)
    v1 = b2 * v + (1.0 - b2) * g * g
    ss = -lr / (1.0 - b1 ** t)
    denom = np.sqrt(v1) / (np.sqrt(1.0 - b2 ** t) * ss) + eps / ss
    return p + m1 / denom, m1, v1


def bc_err(beta, t):
    """Relative error of the kernel's fl(1 - powf(beta, fl32(t))) (module docstring)."""
    t = np.asarray(t, dtype=np.float64)
    x = beta ** t
    tf = np.asarray(t, dtype=np.float32).astype(np.float64)
    shift = abs(math.log(beta)) * np.abs(t - tf) * np.maximum(x, beta ** tf)
    return (POW_ULP * 2 * U * x + POW_ULP * 2.0 ** -149 + shift) / (1.0 - x) + U


def adam_bound(p1, m1, v1, g, m, t, lr, eps_g, b1=B1, b2=B2, eps=EPS, scalar=False):
    """Per-element bounds (E_p, E_m, E_v) of the module docstring; scalar: adam_scalar's extra product roundings."""
    omb1, omb2 = 1.0 - b1, 1.0 - b2
    E_m = omb1 * np.abs(g) * eps_g + (2 if scalar else 1) * U * omb1 * np.abs(g - m) + U * np.abs(m1)
    E_v = omb2 * g * g * (2 * eps_g + eps_g * eps_g) + (3 if scalar else 2) * U * v1
    e_ssn = bc_err(b1, t) + U
    e_c1 = bc_err(b2, t) / 2 + U + e_ssn + U
    e_c2 = e_ssn + U
    with np.errstate(divide="ignore", invalid="ignore"):
        e_sq = np.where(v1 > 0, E_v / np.where(v1 > 0, v1, 1.0) / 2, 0.0) + U
    e_den = np.maximum(e_sq + U + e_c1, e_c2) + U
    ss = -lr / (1.0 - b1 ** t)
    den = np.sqrt(v1) / (np.sqrt(1.0 - b2 ** t) * ss) + eps / ss
    E_p = E_m / np.abs(den) + np.abs(m1 / den) * (e_den + U) + U * np.abs(p1)
    return WIDEN * E_p + FLOOR, WIDEN * E_m + FLOOR, WIDEN * E_v + FLOOR


def polyak_ref(T, p1, tau=TAU):
    return T + tau * (p1 - T)


def polyak_bound(T1, p1, T, E_p, tau=TAU):
    return WIDEN * (tau * E_p + tau * np.abs(p1 - T) * U * (1 + U) + U * np.abs(T1)) + FLOOR


def sumsq_rel(n):
    """Relative bound of b2rl_grad_sumsq over a span of n elements."""
    return WIDEN * ((-(-n // (64 * 256))) + 77) * U


def gscale_ref(G_span, gs, clip, clip_norm, coef_of=None):
    """(gscale, eps_g) per agent [n, 1]: the reference's gradient factor and the kernel's relative error of g * gscale.
    G_span: the agents' gradients over the span b2rl_grad_sumsq covered (clip only). coef_of: agent g takes the clip
    coefficient of agent coef_of[g] (a mistake, for the teeth test)."""
    if not clip:
        return np.full((1, 1), gs), np.full((1, 1), 0.0 if gs == 1.0 else U)
    norm = np.sqrt((G_span.astype(np.float64) ** 2).sum(axis=1, keepdims=True)) * gs
    coef = np.minimum(1.0, clip_norm / (norm + CLIP_EPS))
    if coef_of is not None:
        coef = coef[coef_of]
    eps_c = sumsq_rel(G_span.shape[1]) / 2 + 4 * U
    return gs * coef, np.full((G_span.shape[0], 1), eps_c + 2 * U)


def tf32_lo(x):
    x = np.asarray(x, dtype=np.float32)
    hi = (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    return (x - hi).astype(np.float32)


# ------------------------------------------------------------------------------------------------ test data
def grads(rng, shape):
    """log-uniform magnitudes over 1e-12..1e3, random sign, 5 % exact zeros (fp32)."""
    g = 10.0 ** rng.uniform(-12, 3, shape) * rng.choice([-1.0, 1.0], shape)
    g[rng.random(shape) < 0.05] = 0.0
    return g.astype(np.float32)


def fill_state(rng, arr, sl):
    """arr [n, 5, R] float32: P, T, M, V, G over the columns sl; 5 % of V exactly 0."""
    n, w = arr.shape[0], len(range(*sl.indices(arr.shape[2])))
    p = rng.normal(0.0, 0.1, (n, w))
    arr[:, 0, sl] = p
    arr[:, 1, sl] = p + rng.normal(0.0, 0.01, (n, w))
    arr[:, 2, sl] = 0.1 * grads(rng, (n, w))
    v = grads(rng, (n, w)).astype(np.float64) ** 2
    v[rng.random((n, w)) < 0.05] = 0.0
    arr[:, 3, sl] = v
    arr[:, 4, sl] = grads(rng, (n, w))


class Seg:
    """A b2rl_seg_t on the host side (values as the fp32 the kernel receives)."""

    def __init__(self, begin, end, lr=0.0, adam=False, polyak=False, counter=0, grad_scale=1.0, clip=False):
        self.c = L.Seg(begin, end, lr, int(adam), int(polyak), counter, grad_scale, int(clip))
        self.begin, self.end, self.lr, self.adam, self.polyak = begin, end, self.c.lr, adam, polyak
        self.counter, self.gs, self.clip = counter, self.c.grad_scale, clip


def pairs_of(lay):
    return [(n.off["w2t"], n.off["w2n"]) for n in (*lay.critic, lay.actor)]


def _transpose_span(a, src, dst):
    n = a.shape[0]
    a[:, dst:dst + HH] = a[:, src:src + HH].reshape(n, L.HID, L.HID).transpose(0, 2, 1).reshape(n, HH)


def expect(lay, segs, pre, ctr, clip_norm=0.0, clip_span=None, tau=TAU, b2=B2, eps=EPS, coef_of=None, polyak_pre=False):
    """Reference and bound of one adam_polyak_multi launch from the pre-step arenas pre [n, 5, R] and counters [n, 8]:
    dict key -> (ref, bound, written) over [n, R] for P, T, M, V, G. b2, eps, coef_of, polyak_pre (Polyak with the
    pre-step p) change the reference into a plausible mistake, for the teeth test."""
    n, _, R = pre.shape
    regs = {k: pre[:, r].astype(np.float64) for r, k in enumerate("PTMVG")}
    ref = {k: v.copy() for k, v in regs.items()}
    bnd = {k: np.zeros((n, R)) for k in "PTMVG"}
    wr = {k: np.zeros((n, R), dtype=bool) for k in "PTMVG"}
    for s in segs:
        b, e = s.begin, s.end
        if e <= b:
            continue
        sl = slice(b, e)
        P, T, M, V, G = (regs[k][:, sl] for k in "PTMVG")
        with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
            if s.adam:
                t = ctr[:, s.counter].astype(np.float64)[:, None]
                span = pre[:, 4, clip_span[0]:clip_span[1]] if s.clip else None
                gsc, eps_g = gscale_ref(span, s.gs, s.clip, clip_norm, coef_of)
                g = G * gsc
                p1, m1, v1 = adam_ref(P, g, M, V, t, s.lr, b2=b2, eps=eps)
                E_p, E_m, E_v = adam_bound(p1, m1, v1, g, M, t, s.lr, eps_g, b2=b2, eps=eps)
                for k, x, E in (("P", p1, E_p), ("M", m1, E_m), ("V", v1, E_v)):
                    ref[k][:, sl], bnd[k][:, sl], wr[k][:, sl] = x, E, True
                if s.clip:
                    ref["G"][:, sl], bnd["G"][:, sl], wr["G"][:, sl] = g, WIDEN * np.abs(g) * eps_g + FLOOR, True
            else:
                p1, E_p = P, 0.0
            if s.polyak:
                T1 = polyak_ref(T, P if polyak_pre else p1, tau)
                ref["T"][:, sl], bnd["T"][:, sl], wr["T"][:, sl] = T1, polyak_bound(T1, p1, T, E_p, tau), True
        for src, dst in pairs_of(lay):
            if b <= src < e:  # the shadow: the step computed at w2t, written transposed; its own G is never written
                for k in "PTMV":
                    _transpose_span(ref[k], src, dst)
                    _transpose_span(bnd[k], src, dst)
                wr["G"][:, dst:dst + HH] = False
                ref["G"][:, dst:dst + HH] = regs["G"][:, dst:dst + HH]
    return {k: (ref[k], bnd[k], wr[k]) for k in "PTMVG"}


class Worst:
    def __init__(self):
        self.r = {}

    def add(self, key, ratio):
        self.r[key] = max(self.r.get(key, 0.0), float(ratio))

    def report(self, what=""):
        print(f"{what}: " + ", ".join(f"{k} {v:.3f}" for k, v in sorted(self.r.items())))


def check_within(what, got, ref, bnd, mask, worst=None, key=None):
    got = np.asarray(got, dtype=np.float64)
    g, r, b = got[mask], ref[mask], bnd[mask]
    d = np.abs(g - r)
    bad = ~(d <= b)
    if bad.any():
        i = np.flatnonzero(bad)[:4]
        pos = np.argwhere(mask)[i].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} elements outside the bound; (position, got, ref, bound) "
                             + str([(p, float(g[j]), float(r[j]), float(b[j])) for p, j in zip(pos, i)]))
    ratio = float((d / b).max()) if d.size else 0.0
    if worst is not None:
        worst.add(key or what, ratio)
    return ratio


def check_launch(what, lay, segs, pre, post, ctr, ctr_post, exp, lo_pre=None, lo_post=None, worst=None):
    """post against exp (expect()), everything outside the written sets bitwise unchanged, shadows bitwise w2t^T,
    lo bitwise tf32_lo of what was written, counters untouched."""
    assert np.array_equal(ctr, ctr_post), f"{what}: the launch changed the counters"
    for r, k in enumerate("PTMVG"):
        ref, bnd, wr = exp[k]
        same = post[:, r].view(np.uint32) == pre[:, r].view(np.uint32)
        moved = ~wr & ~same
        assert not moved.any(), f"{what}: region {k} written outside the segments at {np.argwhere(moved)[:4].tolist()}"
        if k == "G":
            check_within(f"{what} G", post[:, r], ref, bnd, wr, worst, "clipped G")
            continue
        check_within(f"{what} {k}", post[:, r], ref, bnd, wr, worst, {"P": "adam p", "T": "polyak T", "M": "adam m",
                                                                       "V": "adam v"}[k])
    for s in segs:
        for src, dst in pairs_of(lay):
            if not (s.begin <= src < s.end):
                continue
            regs = ([0, 2, 3] if s.adam else []) + ([1] if s.polyak else [])
            for r in regs:
                a = post[:, r, src:src + HH].reshape(-1, L.HID, L.HID).transpose(0, 2, 1)
                assert np.array_equal(post[:, r, dst:dst + HH].reshape(-1, L.HID, L.HID).view(np.uint32),
                                      np.ascontiguousarray(a).view(np.uint32)), f"{what}: w2n != w2t^T in region {r}"
    if lo_post is None:
        return
    for h, k in ((0, "P"), (1, "T")):
        wr = exp[k][2]
        want = np.where(wr, tf32_lo(post[:, h]), lo_pre[:, h])
        eq = lo_post[:, h].view(np.uint32) == want.view(np.uint32)
        assert eq.all(), (f"{what}: lo[{h}] differs from tf32_lo of the written values (or was written outside them) at "
                          f"{np.argwhere(~eq)[:4].tolist()}")


# ------------------------------------------------------------------------------------------------ launches
def _lib():
    lib = L.load()
    L.init_device(torch.device("cuda"))
    return lib


def _st():
    return torch.cuda.current_stream().cuda_stream


def adam_args(lay, segs, arena, ctr, sumsq=None, lo=None, clip_norm=0.0, n_agents=None):
    a = L.AdamArgs()
    for i, s in enumerate(segs):
        a.seg[i] = s.c
    a.n_seg, a.n_agents = len(segs), n_agents or arena.shape[0]
    a.polyak, a.clip_norm = TAU, clip_norm
    a.beta1, a.beta2, a.eps = B1, B2, EPS
    a.region_stride, a.arena_agent_stride = lay.region, 5 * lay.region
    a.arena, a.counters, a.grad_sumsq = arena.data_ptr(), ctr.data_ptr(), L.ptr(sumsq)
    a.lo, a.lo_agent_stride = L.ptr(lo), 2 * lay.region
    set_shadow_pairs(a, lay)
    return a


def seg_union(segs, R):
    m = np.zeros(R, dtype=bool)
    for s in segs:
        m[s.begin:s.end] = True
    return m


def prepare(lay, segs, n, rng):
    """Host arenas [n, 5, R]: the sentinel outside the segments, random state inside, NaN in every region of the shadows
    (w2n) of the pairs a segment holds."""
    R = lay.region
    pre = np.full((n, 5, R), SENT, dtype=np.float32)
    m = seg_union(segs, R)
    edges = np.flatnonzero(np.diff(np.concatenate([[0], m.astype(np.int8), [0]])))
    for b, e in zip(edges[::2], edges[1::2]):
        fill_state(rng, pre, slice(int(b), int(e)))
    for src, dst in pairs_of(lay):
        if m[src]:
            pre[:, :, dst:dst + HH] = QNAN
    return pre


def run_adam(lib, lay, segs, pre, ctr_np, lo=False, clip_norm=0.0, clip_span=None):
    """Upload, (b2rl_grad_sumsq over clip_span,) one adam_polyak_multi launch, read back."""
    n, R = pre.shape[0], lay.region
    arena = torch.from_numpy(pre).cuda()
    ctr = torch.from_numpy(ctr_np).cuda()
    sumsq = torch.zeros(n, device="cuda")
    scratch = torch.zeros(n * 64, device="cuda")
    lo_pre = np.full((n, 2, R), SENT, dtype=np.float32)
    lo_t = torch.from_numpy(lo_pre).cuda() if lo else None
    if clip_span is not None:
        L.check(lib.b2rl_grad_sumsq(arena.data_ptr(), R, 5 * R, clip_span[0], clip_span[1], n, sumsq.data_ptr(),
                                    scratch.data_ptr(), _st()), "grad_sumsq")
    a = adam_args(lay, segs, arena, ctr, sumsq, lo_t, clip_norm)
    L.check(lib.b2rl_adam_polyak_multi(C.byref(a), _st()), "adam_polyak_multi")
    torch.cuda.synchronize()
    return (arena.cpu().numpy(), ctr.cpu().numpy(), sumsq.cpu().numpy(), lo_pre if lo else None,
            lo_t.cpu().numpy() if lo else None)


def counters_for(n, rng, q, pi=None):
    ctr = rng.integers(0, 2 ** 40, (n, 8)).astype(np.int64)
    ctr[:, L.CTR_Q] = q
    ctr[:, L.CTR_PI] = pi if pi is not None else q[::-1]
    return ctr


# ------------------------------------------------------------------------------------------------ 1. adam_polyak_multi
LAYOUTS = [(11, 3, False, True), (376, 17, False, True), (27, 8, True, True), (5, 2, False, False), (1, 1, True, False)]
LR_Q, LR_PI = f32(1e-3), f32(3e-4)


def segsets(lay):
    c0, c1, a = lay.critic[0], lay.critic[1], lay.actor
    Q = lambda pol: Seg(c0.begin, c1.end, LR_Q, adam=True, polyak=pol, counter=L.CTR_Q)
    PI = lambda pol, clip: Seg(a.begin, a.end, LR_PI, adam=True, polyak=pol, counter=L.CTR_PI, clip=clip)
    free = []  # 8 pair-free spans: around every net's w2t, the second piece of each net split once more
    for n in (c0, c1, a):
        w = n.off["w2t"]
        free.append((n.begin, w))
        mid = w + HH + ((n.core_end - w - HH) // 8) * 4
        free += [(w + HH, mid), (mid, n.core_end)]
    free = free[:8]
    mid0 = c0.begin + (c0.off["b1"] - c0.begin) // 8 * 4  # inside critic 0's first weight
    return {
        "critic": [Q(False)],
        "critic+polyak": [Q(True)],
        "actor": [PI(False, False)],
        "actor+polyak+clip": [PI(True, True)],
        "polyak critics+actor": [Seg(c0.begin, c1.end, polyak=True), Seg(a.begin, a.end, polyak=True)],
        "td3 critic step without actor update": [Q(True), Seg(a.begin, a.end, polyak=True)],
        "8 pair-free segments": [Seg(b, e, f32(10.0 ** -(2 + i % 3)), adam=i % 3 != 2, polyak=i % 2 == 0,
                                     counter=i % 2) for i, (b, e) in enumerate(free)],
        "boundary inside a tensor": [Seg(c0.begin, mid0, LR_PI, adam=True, counter=L.CTR_PI),
                                     Seg(mid0, c1.end, LR_Q, adam=True, polyak=True, counter=L.CTR_Q)],
        "zero-length segment": [Seg(a.begin, a.begin, LR_Q, adam=True, polyak=True), Q(False),
                                Seg(c1.end, c1.end, polyak=True)],
        "critic and actor, two counters": [Q(True), PI(False, False)],
    }


@pytest.mark.gpu
@pytest.mark.parametrize("ob,ac,td3,ln", LAYOUTS)
def test_adam_polyak_multi_matches_float64(ob, ac, td3, ln):
    """One launch per segment set and mirror option; 7 stacked agents, one per step count (the actor's counter runs the
    other way round, so two Adam segments of one launch see different t)."""
    lib = _lib()
    lay = make_layout(ob, ac, td3, ln)
    rng = np.random.default_rng(ob * 1000 + ac)
    worst = Worst()
    q = np.array(TS, dtype=np.int64)
    for name, segs in segsets(lay).items():
        pre = prepare(lay, segs, len(TS), rng)
        ctr = counters_for(len(TS), rng, q)
        clip = any(s.clip for s in segs)
        span = (lay.actor.begin, lay.actor.core_end) if clip else None
        clip_norm = f32(1.0) if clip else 0.0
        exp = expect(lay, segs, pre, ctr, clip_norm, span)
        for lo in (False, True):  # (the same pre-step state twice)
            post, ctr_post, sumsq, lo_pre, lo_post = run_adam(lib, lay, segs, pre, ctr, lo, clip_norm, span)
            if clip:
                want = (pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1)
                check_within(f"{name} sumsq", sumsq, want, sumsq_rel(span[1] - span[0]) * want + FLOOR,
                             np.ones_like(want, dtype=bool), worst, "sumsq")
            check_launch(f"({ob},{ac},{'td3' if td3 else 'sac'},{'ln' if ln else 'noln'}) {name} lo={lo}", lay, segs,
                         pre, post, ctr, ctr_post, exp, lo_pre, lo_post, worst)
    worst.report(f"adam_polyak_multi ({ob},{ac}) worst dev/bound")


# ------------------------------------------------------------------------------------------------ 2. many steps
@pytest.mark.gpu
def test_adam_200_critic_steps_each_within_the_local_bound():
    """t = 1..200 on the SAC Hopper layout: b2rl_bump_counter then Adam + Polyak over the critics; every step is checked
    from the state the previous one left (fresh gradients each step)."""
    lib = _lib()
    lay = make_layout(11, 3, False, True)
    R, rng, worst = lay.region, np.random.default_rng(200), Worst()
    segs = [Seg(lay.critic[0].begin, lay.critic[1].end, LR_Q, adam=True, polyak=True, counter=L.CTR_Q)]
    pre = prepare(lay, segs, 1, rng)
    b, e = segs[0].begin, segs[0].end
    own = np.ones(e - b, dtype=bool)  # (not the shadows, which stay NaN in G, M and V)
    for src, dst in pairs_of(lay):
        if b <= src < e:
            own[dst - b:dst - b + HH] = False
    pre[:, 2:4, b:e][:, :, own] = 0.0  # Adam starts from zero moments
    arena = torch.from_numpy(pre).cuda()
    ctr = torch.zeros(1, 8, dtype=torch.int64, device="cuda")
    a = adam_args(lay, segs, arena, ctr)
    for t in range(1, 201):
        g = grads(rng, (1, e - b))
        g[:, ~own] = QNAN
        arena[:, 4, b:e] = torch.from_numpy(g).cuda()
        torch.cuda.synchronize()
        before, c0 = arena.cpu().numpy(), ctr.cpu().numpy()
        L.check(lib.b2rl_bump_counter(ctr.data_ptr(), L.CTR_Q, 1, _st()), "bump_counter")
        L.check(lib.b2rl_adam_polyak_multi(C.byref(a), _st()), "adam_polyak_multi")
        torch.cuda.synchronize()
        after, c1 = arena.cpu().numpy(), ctr.cpu().numpy()
        want = c0.copy()
        want[0, L.CTR_Q] += 1
        assert np.array_equal(c1, want) and c1[0, L.CTR_Q] == t
        check_launch(f"step {t}", lay, segs, before, after, c1, c1, expect(lay, segs, before, c1), worst=worst)
    worst.report("200 critic steps worst dev/bound")


# ------------------------------------------------------------------------------------------------ 3. clipping, sumsq
@pytest.mark.gpu
def test_grad_sumsq_matches_float64():
    lib = _lib()
    worst = Worst()
    spans = [(1, 2), (5, 5), (0, 64 * 256 * 8 + 4 * 1234 + 1)]
    for ob, ac, td3, ln in LAYOUTS:
        lay = make_layout(ob, ac, td3, ln)
        spans.append((lay.actor.begin, lay.actor.core_end))
    R = max(e for _, e in spans) + 16
    n = 3
    rng = np.random.default_rng(5)
    host = np.zeros((n, 5, R), dtype=np.float32)
    host[:, 4] = grads(rng, (n, R))
    arena = torch.from_numpy(host).cuda()
    sumsq = torch.full((n,), 7.0, device="cuda")
    scratch = torch.zeros(n * 64, device="cuda")
    for b, e in spans:
        L.check(lib.b2rl_grad_sumsq(arena.data_ptr(), R, 5 * R, b, e, n, sumsq.data_ptr(), scratch.data_ptr(), _st()), "sumsq")
        got = sumsq.cpu().numpy()
        want = (host[:, 4, b:e].astype(np.float64) ** 2).sum(axis=1)
        if e == b:
            assert np.array_equal(got, np.zeros(n, dtype=np.float32)), got
            continue
        check_within(f"sumsq [{b},{e})", got, want, sumsq_rel(e - b) * want + FLOOR, np.ones(n, dtype=bool), worst, "sumsq")
    worst.report("grad_sumsq worst dev/bound")


@pytest.mark.gpu
@pytest.mark.parametrize("grad_scale", [1.0, 0.5, 1.0 / 3.0])
@pytest.mark.parametrize("clip", [False, True])
def test_clip_and_grad_scale_per_agent(grad_scale, clip):
    """Five agents, each with its own gradient norm and step count: norm << clip, clip (1 -/+ 1e-3), norm >> clip and an
    all-zero gradient (coefficient 1, no NaN). Each agent is judged against its own reference."""
    lib = _lib()
    lay = make_layout(11, 3, False, True)
    a = lay.actor
    span = (a.begin, a.core_end)
    segs = [Seg(a.begin, a.end, LR_PI, adam=True, polyak=True, counter=L.CTR_PI, grad_scale=grad_scale, clip=clip)]
    rng = np.random.default_rng(31)
    n, clip_norm = 5, f32(2.5)
    pre = prepare(lay, segs, n, rng)
    gsc = f32(grad_scale)
    norm = np.sqrt((pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1)) * gsc
    target = np.array([1e-3, 1 - 1e-3, 1 + 1e-3, 1e3, 0.0]) * clip_norm
    pre[:, 4, span[0]:span[1]] = (pre[:, 4, span[0]:span[1]] * (target / norm)[:, None]).astype(np.float32)
    ctr = counters_for(n, rng, np.array([5, 6, 7, 8, 9]), np.array([1, 2, 1000, 2 ** 24 + 1, 3]))
    post, ctr_post, sumsq, _, _ = run_adam(lib, lay, segs, pre, ctr, False, clip_norm, span if clip else None)
    assert np.isfinite(post[:, :4, a.begin:a.end]).all()
    exp = expect(lay, segs, pre, ctr, clip_norm, span)
    worst = Worst()
    check_launch(f"clip={clip} grad_scale={grad_scale}", lay, segs, pre, post, ctr, ctr_post, exp, worst=worst)
    if clip:
        norm = np.sqrt((pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1)) * gsc
        coef = np.minimum(1.0, clip_norm / (norm + CLIP_EPS))
        assert coef[0] == 1.0 and coef[1] == 1.0 and coef[2] < 1.0 and coef[3] < 1e-2 and coef[4] == 1.0, coef
    worst.report(f"clip={clip} grad_scale={grad_scale:.3f} worst dev/bound")


# ------------------------------------------------------------------------------------------------ 4. fused optimizer
def _population(td3, seed=42):
    from oracle import make_synthetic_transitions
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.population import Population
    hps = (td3_hps if td3 else sac_hps)(batch_size=32)
    pop = Population([0, 1, 2], 11, 3, [-1.0] * 3, [1.0] * 3, hps, "cuda", seed=seed, rb_capacity=500, use_graphs=False)
    pop.fill_replay(make_synthetic_transitions(400, 11, 3, [-1.0] * 3, [1.0] * 3, seed=9))
    return pop


def _pop_opt(pop, segs):
    return adam_args(pop.layout, segs, pop.arena.flat, pop.counters, pop.sumsq, None, 0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("td3", [False, True])
def test_fused_optimizer_stacked_high_counters_bitwise(td3):
    """b2rl_{critic,actor}_update_opt on one row-path Population (N = 3) against the kernel + adam_polyak_multi on an
    identically seeded twin, at step counts {1, 7, 1000} and {2^24 + 1, 2^32 + 5, 2^40}, with and without an extra
    Polyak-only segment: bitwise-equal arenas, counters and log blocks."""
    lib = _lib()
    fused, ref = _population(td3), _population(td3)
    lay, st = fused.layout, _st()
    c0, c1, a = lay.critic[0], lay.critic[1], lay.actor
    for ts in ((1, 7, 1000), (2 ** 24 + 1, 2 ** 32 + 5, 2 ** 40)):
        for extra in (False, True):
            for pop in (fused, ref):
                pop.counters[:, L.CTR_Q] = torch.tensor(ts, device="cuda") - 1  # the step bumps them to t first
                pop.counters[:, L.CTR_PI] = torch.tensor(ts[::-1], device="cuda") - 1
            q_segs = [Seg(c0.begin, c1.end, f32(fused.hps.qnets_lr), adam=True, polyak=True, counter=L.CTR_Q)]
            q_segs += [Seg(a.begin, a.end, polyak=True)] if extra else []
            pi_segs = [Seg(a.begin, a.end, f32(fused.hps.actor_lr), adam=True, polyak=extra, counter=L.CTR_PI)]
            for pop in (fused, ref):
                L.check(lib.b2rl_replay_sample_gather(
                    pop.storage.data_ptr(), pop.storage[0].numel(), 0, pop.fmt, pop.B, pop.N, None, pop.idx.data_ptr(),
                    pop.rows.data_ptr(), C.c_uint64(pop.seed), pop.counters.data_ptr(), L.CTR_Q, 0, pop.base, st), "gather")
            L.check(lib.b2rl_critic_update_opt(C.byref(fused.args), C.byref(_pop_opt(fused, q_segs)), st), "critic_update_opt")
            L.check((lib.b2rl_critic_update_td3 if td3 else lib.b2rl_critic_update_sac)(C.byref(ref.args), st), "critic")
            L.check(lib.b2rl_adam_polyak_multi(C.byref(_pop_opt(ref, q_segs)), st), "adam")
            L.check(lib.b2rl_actor_update_opt(C.byref(fused.args), C.byref(_pop_opt(fused, pi_segs)), st), "actor_update_opt")
            L.check((lib.b2rl_actor_update_td3 if td3 else lib.b2rl_actor_update_sac)(C.byref(ref.args), st), "actor")
            L.check(lib.b2rl_adam_polyak_multi(C.byref(_pop_opt(ref, pi_segs)), st), "adam")
            torch.cuda.synchronize()
            tag = f"t={ts} extra={extra}"
            assert torch.equal(fused.arena.flat, ref.arena.flat), f"{tag}: fused optimizer differs from adam_polyak_multi"
            assert torch.equal(fused.counters, ref.counters), tag
            assert torch.equal(fused.out, ref.out), tag
            assert fused.counters[:, L.CTR_Q].tolist() == list(ts), tag
            assert torch.isfinite(fused.arena.flat[:, :4]).all(), tag


# ------------------------------------------------------------------------------------------------ 5. temperature Adam
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 128, 129, 300])
@pytest.mark.parametrize("grad_scale,table", [(1.0, False), (0.5, False), (1.0, True)], ids=["1.0", "0.5", "1.0-table"])
def test_alpha_adam_matches_float64(n, grad_scale, table):
    """One temperature Adam step per agent (b2rl_alpha_adam); table: each agent's own lr from a per-agent hyperparameter
    table (b2rl_alpha_adam_hp)."""
    lib = _lib()
    rng = np.random.default_rng(n)
    st = np.zeros((n, 5), dtype=np.float32)
    st[:, 0] = rng.normal(0.0, 1.0, n)
    st[:, 1] = grads(rng, n)
    st[:, 2] = 0.1 * grads(rng, n)
    st[:, 3] = grads(rng, n).astype(np.float64) ** 2
    st[rng.random(n) < 0.1, 3] = 0.0
    st[:, 4] = SENT
    ctr = rng.integers(0, 2 ** 40, (n, 8)).astype(np.int64)
    ts = np.array([(1, 2, 1000, 2 ** 24 + 1)[i % 4] for i in range(n)], dtype=np.int64)
    ctr[:, L.CTR_ALPHA] = ts - 1
    out0 = np.full((n, 8), SENT, dtype=np.float32)
    d_st, d_ctr, d_out = (torch.from_numpy(x).cuda() for x in (st, ctr, out0))
    lr = f32(1e-3)
    if table:
        hp = np.zeros((n, C.sizeof(L.AgentHp) // 4), dtype=np.float32)
        hp[:, L.CTR_ALPHA] = np.array([1e-4, 3e-3, 0.05], dtype=np.float32)[np.arange(n) % 3]
        d_hp = torch.from_numpy(hp).cuda()
        lr = hp[:, L.CTR_ALPHA].astype(np.float64)
        L.check(lib.b2rl_alpha_adam_hp(d_st.data_ptr(), d_ctr.data_ptr(), n, d_hp.data_ptr(), grad_scale, d_out.data_ptr(), _st()),
                "alpha_adam_hp")
    else:
        L.check(lib.b2rl_alpha_adam(d_st.data_ptr(), d_ctr.data_ptr(), n, lr, grad_scale, d_out.data_ptr(), _st()), "alpha_adam")
    torch.cuda.synchronize()
    got, c1, out = d_st.cpu().numpy(), d_ctr.cpu().numpy(), d_out.cpu().numpy()
    want = ctr.copy()
    want[:, L.CTR_ALPHA] += 1
    assert np.array_equal(c1, want), "alpha_adam must advance counters[ALPHA] by one and touch nothing else"
    gs = f32(grad_scale)
    x = st.astype(np.float64)
    g = x[:, 1] * gs
    t = ts.astype(np.float64)
    p1, m1, v1 = adam_ref(x[:, 0], g, x[:, 2], x[:, 3], t, lr)
    E_p, E_m, E_v = adam_bound(p1, m1, v1, g, x[:, 2], t, lr, 0.0 if gs == 1.0 else U, scalar=True)
    worst = Worst()
    every = np.ones(n, dtype=bool)
    check_within("log_alpha", got[:, 0], p1, E_p, every, worst, "alpha p")
    check_within("exp_avg", got[:, 2], m1, E_m, every, worst, "alpha m")
    check_within("exp_avg_sq", got[:, 3], v1, E_v, every, worst, "alpha v")
    assert np.array_equal(got[:, 1], g.astype(np.float32)), "state[1] must hold the scaled gradient"
    assert np.array_equal(got[:, 4].view(np.uint32), st[:, 4].view(np.uint32)), "state[4] must stay untouched"
    assert np.array_equal(out[:, L.OUT_ALPHA_LOSS].view(np.uint32), got[:, 1].view(np.uint32))
    with np.errstate(over="ignore"):
        alpha = np.exp(got[:, 0].astype(np.float64))
    fin = alpha < 2.0 ** 127  # (the random moments take some log_alpha far out: expf overflows beyond 2^128)
    check_within("out[ALPHA]", out[:, L.OUT_ALPHA], alpha, (2 * EXP_ULP + 1) * U * alpha + 2.0 ** -148, fin, worst, "alpha exp")
    assert np.isinf(out[alpha >= 2.0 ** 128, L.OUT_ALPHA]).all()
    keep = [i for i in range(8) if i not in (L.OUT_ALPHA_LOSS, L.OUT_ALPHA)]
    assert np.array_equal(out[:, keep].view(np.uint32), out0[:, keep].view(np.uint32))
    worst.report(f"alpha_adam n={n} grad_scale={grad_scale} table={table} worst dev/bound")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 128, 129])
def test_bump_counter_moves_one_slot(n):
    lib = _lib()
    rng = np.random.default_rng(n + 1)
    ctr = rng.integers(0, 2 ** 62, (n, 8)).astype(np.int64)
    d = torch.from_numpy(ctr).cuda()
    for which in (L.CTR_Q, L.CTR_ALPHA, L.CTR_XTICKET):
        L.check(lib.b2rl_bump_counter(d.data_ptr(), which, n, _st()), "bump_counter")
        torch.cuda.synchronize()
        ctr[:, which] += 1
        assert np.array_equal(d.cpu().numpy(), ctr), f"bump_counter(which={which}, n={n})"


# ------------------------------------------------------------------------------------------------ 6. large offsets
@pytest.mark.gpu
def test_offsets_beyond_2_31_floats():
    """1100 stacked SAC Hopper agents (2 049 360 floats each: agents from 1048 on start beyond 2^31 floats): one
    grad_sumsq and one adam_polyak_multi launch over all of them, agents {0, 1047, 1048, 1099} checked."""
    lay = make_layout(11, 3, False, True)
    n, R = 1100, lay.region
    assert 5 * R == 2049360 and 1048 * 5 * R >= 2 ** 31 > 1047 * 5 * R
    if torch.cuda.mem_get_info()[0] < 16 * 2 ** 30:
        pytest.skip("needs 16 GB of free device memory")
    lib = _lib()
    c0, c1, a = lay.critic[0], lay.critic[1], lay.actor
    segs = [Seg(c0.begin, c1.end, LR_Q, adam=True, polyak=True, counter=L.CTR_Q),
            Seg(a.begin, a.end, LR_PI, adam=True, counter=L.CTR_PI, clip=True)]
    span = (a.begin, a.core_end)
    pick = [0, 1047, 1048, 1099]
    rng = np.random.default_rng(1100)
    pre = prepare(lay, segs, len(pick), rng)
    ctr = counters_for(len(pick), rng, np.array([1, 1000, 3, 2 ** 24 + 1]))
    arena = torch.zeros(n, 5, R, device="cuda")
    counters = torch.ones(n, 8, dtype=torch.int64, device="cuda")
    sumsq = torch.zeros(n, device="cuda")
    scratch = torch.zeros(n * 64, device="cuda")
    idx = torch.tensor(pick, device="cuda")
    arena[idx] = torch.from_numpy(pre).cuda()
    counters[idx] = torch.from_numpy(ctr).cuda()
    clip_norm = f32(1.0)
    try:
        L.check(lib.b2rl_grad_sumsq(arena.data_ptr(), R, 5 * R, span[0], span[1], n, sumsq.data_ptr(), scratch.data_ptr(),
                                    _st()), "grad_sumsq")
        L.check(lib.b2rl_adam_polyak_multi(C.byref(adam_args(lay, segs, arena, counters, sumsq, None, clip_norm)), _st()),
                "adam_polyak_multi")
        torch.cuda.synchronize()
        post, ctr_post, ss = arena[idx].cpu().numpy(), counters[idx].cpu().numpy(), sumsq[idx].cpu().numpy()
    finally:
        del arena
        torch.cuda.empty_cache()
    want = (pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1)
    worst = Worst()
    check_within("sumsq", ss, want, sumsq_rel(span[1] - span[0]) * want + FLOOR, np.ones(len(pick), dtype=bool), worst, "sumsq")
    check_launch("1100 agents", lay, segs, pre, post, ctr, ctr_post, expect(lay, segs, pre, ctr, clip_norm, span), worst=worst)
    worst.report("agents 0/1047/1048/1099 worst dev/bound")


# ------------------------------------------------------------------------------------------------ 7. fused path + mirror
def _engine_agent():
    from tests.golden.cases import case_inputs
    from tests.helpers import make_agent
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    inp = case_inputs("sac_hopper")
    ag = make_agent(inp, seed=5)
    td = inp["storage"]
    rb = ReplayBuffer(td["observations"].shape[0], "cuda", seed=5)
    rb.extend({k: v.cuda() for k, v in td.items()})
    return ag, rb


@pytest.mark.gpu
def test_fused_engine_keeps_the_lo_mirror_current():
    """An agent with a 3xTF32 mirror in a LearnerEngine(fused_opt=True): the mirror must equal tf32_lo of the online and
    target regions after an iteration (the fused weight-gradient optimizer does not write it, so the step must take the
    three-launch form), and the result must equal a fused_opt=False engine's, launch count included."""
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    (ag, rb), (ag2, rb2) = _engine_agent(), _engine_agent()
    for x in (ag, ag2):
        x.lo_mirror()
    eng = LearnerEngine(ag, rb, use_graphs=False, fused_opt=True)
    eng2 = LearnerEngine(ag2, rb2, use_graphs=False, fused_opt=False)
    for i in range(2):
        eng.iteration(i)
        eng2.iteration(i)
    torch.cuda.synchronize()
    flat = ag.arena.flat[0, :2].cpu().numpy()
    lo = ag._lo[0].cpu().numpy()
    stale = int((lo.view(np.uint32) != tf32_lo(flat).view(np.uint32)).sum())
    assert stale == 0, f"{stale} elements of the lo mirror differ from tf32_lo of the parameters after a fused-optimizer iteration"
    assert torch.equal(ag.arena.flat, ag2.arena.flat) and torch.equal(ag._lo, ag2._lo)
    assert eng.launches_per_variant == eng2.launches_per_variant


@pytest.mark.gpu
def test_fused_entry_points_refuse_a_lo_mirror():
    lib = _lib()
    ag, _ = _engine_agent()
    ag.lo_mirror()
    rows = torch.zeros(ag.batch_size, ag.fmt.row_stride, device="cuda")
    args = ag.update_args(rows)
    torch.cuda.synchronize()
    flat, ctr, lo = ag.arena.flat.clone(), ag.counters.clone(), ag._lo.clone()
    for fn, segs in ((lib.b2rl_critic_update_opt, ag.critic_segs(True)), (lib.b2rl_actor_update_opt, ag.actor_segs(False))):
        opt = ag._adam_args(segs)
        assert opt.lo
        assert fn(C.byref(args), C.byref(opt), _st()) == -1  # B2RL_E_INVALID
        assert b"lo mirror" in lib.b2rl_last_error()
    torch.cuda.synchronize()
    assert torch.equal(ag.arena.flat, flat) and torch.equal(ag.counters, ctr) and torch.equal(ag._lo, lo), "a refused call launched"


# ------------------------------------------------------------------------------------------------ 8. the oracle's Adam
def _oracle_vs_torch(device, capturable, dtype):
    from oracle.sac_td3_oracle import _Adam
    g = torch.Generator().manual_seed(3)
    init = [torch.randn(7, 5, generator=g, dtype=torch.float64), torch.randn(11, generator=g, dtype=torch.float64)]
    mine = [p.to(device, dtype).clone() for p in init]
    theirs = [p.to(device, dtype).clone().requires_grad_(True) for p in init]
    opt = _Adam(mine, lr=3e-4, capturable=capturable)
    topt = torch.optim.Adam(theirs, lr=3e-4, capturable=capturable, foreach=False)
    for _ in range(5):
        for p, q in zip(mine, theirs):
            gr = (torch.randn(p.shape, generator=g, dtype=torch.float64) * 10.0 ** float(torch.randint(-6, 2, (1,), generator=g)))
            p.grad = gr.to(device, dtype)
            q.grad = gr.to(device, dtype)
        opt.step()
        topt.step()
        for p, q in zip(mine, theirs):
            d = float((p.detach().double() - q.detach().double()).abs().max() / q.detach().double().abs().max())
            assert d <= (1e-13 if dtype == torch.float64 else 1e-6), d


def test_oracle_adam_matches_torch():
    """oracle._Adam (capturable=False) against torch.optim.Adam over 5 steps, float64 and float32."""
    _oracle_vs_torch("cpu", False, torch.float64)
    _oracle_vs_torch("cpu", False, torch.float32)


@pytest.mark.gpu
def test_oracle_adam_capturable_matches_torch():
    _oracle_vs_torch("cuda", True, torch.float32)


# ------------------------------------------------------------------------------------------------ teeth (CPU)
def _emulate(lay, segs, pre, ctr, clip_norm, span):
    """fp32 numpy emulation of adam_polyak_multi (an fma: one rounding of the exact float64 result; powf: numpy's)."""
    f = np.float32
    fma = lambda a, b, c: (np.float64(a) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(f)
    post = pre.copy()
    for s in segs:
        sl = slice(s.begin, s.end)
        P, T, M, V, G = (pre[:, r, sl] for r in range(5))
        p1 = P
        with np.errstate(invalid="ignore"):
            if s.adam:
                t = ctr[:, s.counter].astype(f)[:, None]
                bc1, bc2 = f(1) - np.power(f(B1), t), f(1) - np.power(f(B2), t)
                ssn = -(f(s.lr) / bc1)
                c1, c2 = np.sqrt(bc2) * ssn, f(EPS) / ssn
                gs = np.full((pre.shape[0], 1), f(s.gs))
                if s.clip:
                    ss = (pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1, keepdims=True).astype(f)
                    gs = gs * np.minimum(f(1), f(clip_norm) / (np.sqrt(ss) * f(s.gs) + f(CLIP_EPS)))
                g = G * gs
                m1 = fma(f(1) - f(B1), g - M, M)
                v1 = fma(f(1) - f(B2), g * g, V * f(B2))  # (the kernel rounds (1 - b2) g instead: same bound)
                p1 = P + m1 / (np.sqrt(v1) / c1 + c2)
                post[:, 0, sl], post[:, 2, sl], post[:, 3, sl] = p1, m1, v1
                if s.clip:
                    post[:, 4, sl] = g
            if s.polyak:
                post[:, 1, sl] = fma(f(TAU), p1 - T, T)
        for src, dst in pairs_of(lay):
            if s.begin <= src < s.end:  # the shadow tiles
                post[:, 4, dst:dst + HH] = pre[:, 4, dst:dst + HH]
                for r in ([0, 2, 3] if s.adam else []) + ([1] if s.polyak else []):
                    post[:, r, dst:dst + HH] = post[:, r, src:src + HH].reshape(-1, L.HID, L.HID).transpose(0, 2, 1).reshape(-1, HH)
    return post


def _worst_ratio(exp, vals, keys="PTMVG"):
    """max |vals - ref| / bound over the written elements; vals: key -> [n, R]."""
    r = 0.0
    for k in keys:
        ref, bnd, wr = exp[k]
        with np.errstate(invalid="ignore"):
            d = np.abs(np.asarray(vals[k], np.float64) - ref)[wr] / bnd[wr]
        if d.size:
            r = max(r, float(np.nan_to_num(d, nan=np.inf).max()))
    return r


def test_bound_has_teeth():
    """On data drawn like the GPU tests' (four agents at t = 2, 3, 10, 1000 with clip coefficients 1 ... 1e-3, grad_scale
    0.5), an fp32 emulation of the kernel stays within the bound, and each of these mistakes exceeds it at least tenfold
    somewhere: t - 1 for t, beta2 = 0.99, eps dropped, Polyak with the pre-step p, grad_scale ignored, two agents' step
    counters swapped, the clip coefficient of another agent."""
    lay = make_layout(5, 2, False, False)
    a = lay.actor
    span = (a.begin, a.core_end)
    clip_norm, rng = f32(2.5), np.random.default_rng(11)
    seg = lambda gs: [Seg(a.begin, a.end, LR_PI, adam=True, polyak=True, counter=L.CTR_PI, grad_scale=gs, clip=True)]
    segs = seg(0.5)
    pre = prepare(lay, segs, 4, rng)
    norm = np.sqrt((pre[:, 4, span[0]:span[1]].astype(np.float64) ** 2).sum(axis=1)) * 0.5
    pre[:, 4, span[0]:span[1]] *= (np.array([1e-3, 1.0, 10.0, 1e3]) * clip_norm / norm)[:, None].astype(np.float32)
    ctr = counters_for(4, rng, np.array([1, 1, 1, 1]), np.array([2, 3, 10, 1000]))
    exp = expect(lay, segs, pre, ctr, clip_norm, span)
    post = _emulate(lay, segs, pre, ctr, clip_norm, span)
    good = _worst_ratio(exp, {k: post[:, r] for r, k in enumerate("PTMVG")})
    print(f"fp32 emulation: worst dev/bound {good:.3f}")
    assert good <= 1.0, "a correct fp32 implementation must stay within the bound"

    def exceeds(name, **kw):
        wrong = expect(lay, kw.pop("segs", segs), pre, kw.pop("ctr", ctr), clip_norm, span, **kw)
        r = _worst_ratio(exp, {k: wrong[k][0] for k in "PTMVG"})
        print(f"{name}: worst dev/bound {r:.3g}")
        assert r >= 10.0, f"{name} stays within {r:.3g} x the bound"

    c = ctr.copy()
    c[:, L.CTR_PI] -= 1
    exceeds("t - 1 for t", ctr=c)
    exceeds("beta2 = 0.99", b2=f32(0.99))
    exceeds("eps dropped", eps=0.0)
    exceeds("Polyak with the pre-step p", polyak_pre=True)
    exceeds("grad_scale ignored", segs=seg(1.0))
    c = ctr.copy()
    c[[0, 1], L.CTR_PI] = c[[1, 0], L.CTR_PI]
    exceeds("two agents' step counters swapped", ctr=c)
    exceeds("the clip coefficient of another agent", coef_of=[1, 0, 3, 2])
