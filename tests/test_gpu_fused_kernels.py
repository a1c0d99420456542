"""The row-group learner's fused kernels — critic_fused (csrc/critic.cu), actor_fused and alpha_kernel (csrc/actor.cu) —
each launched on its own (b2rl_launch_single) on hand-filled inputs, every per-row output against a float64 restatement
of the same arithmetic, element by element, on every row: no row is set aside for lying near a ReLU kink.

Bounds follow test_gpu_wide_kernels.py (u = 2^-24; gamma_k = k u / (1 - k u) over sum|terms|; the running error class R,
whose inputs may carry their own bounds, which then propagate). k from the loop structure of csrc/mlp_cluster.cuh:
  first layer (first_smem / first_global, reduce_slice)   ceil(K/8) FMAs per warp, 7 partial adds, the bias  k = ceil(K/8) + 8
  hidden layer (hidden_fma, reduce_slice)                  32 FMAs per warp, 7 partial adds, the bias        k = 40
  dX product through w2n (no bias)                                                                           k = 39
  heads, dQ/da (rowdot)                                    8 FMAs per lane + 5 shuffle levels (+ the bias)   k = 14 / 13
  LayerNorm statistics (row_stats)                         3-level tree + 5 shuffle levels                   k = 8
                                                           two-pass variance: 8 FMAs + 5 shuffle levels      k = 13
                                                           sqrtf and the division are correctly rounded (no fast-math)
  actor head backward (dLoss/dh2)                          a chain of out_dim FMAs                           k = out_dim
  per-tile partials (8 rows in sequence from 0)                                                              k = 7
  PART_DB3 of the actor (((d0+d1)+(d2+d3))+((d4+d5)+(d6+d7)))                                                k = 3
  tanhf / expf / logf: 2 / 2 / 1 ulp (CUDA C++ Programming Guide), as in policy_head_ref.
A bound carried forward |W|-wise through several 256-wide layers loses the weights' signs and soon accepts anything, so:
  - every stage the kernel stores (workspace h1 / h2 / dz1 / dz2 / dZ3, Q, y) is checked from the kernel's own stored input
    of that stage (h2 from its h1, Q from its h2, dZ3 from its Q and y, dz2 from its dZ3, dz1 from its dz2): each bound
    stays tight, and the chain of stages still covers the whole kernel;
  - the per-row scalars of passes that store nothing (the TD target; the next action and log pi feeding it; alpha_kernel's
    log pi) also get a first-order bound by sensitivities (class Sens: every rounding's local bound times |d output / d that
    rounding|, one backward pass), and the smaller of the two bounds is used;
  - the critic passes inside the actor step keep the R bound, with the widened masks below.
ReLU is 1-Lipschitz: a forward bound passes through it unchanged, and the reference never has to agree with the kernel on
which side of a kink a unit lies. The backward pass needs the mask:
  - where the kernel stored the activations (the online critic k of the critic step, workspace slot k; the actor of the
    actor step, slot 0), the kernel's own mask h > 0 — exactly the `on` that layer_bwd_rows recomputes. Wherever it
    differs from the float64 mask, the float64 pre-activation must lie within its own forward bound of zero;
  - where it did not (the critic passes inside the actor step), a unit whose |pre-activation| is within its bound takes
    the mask R(0.5, 0.5) — either value — and every other unit its float64 mask. SAC's arg-min of Q_0, Q_1 is treated the
    same way when |Q_0 - Q_1| is within their bounds.
The share of units whose mask had to be widened is reported. Saturated tanh samples (|1 - y^2| < 1e-3) are reported
apart, as in test_gpu_wide_kernels.py.

The noise the kernels used (eps_out / eps2_out) is the reference's noise; device-drawn noise (eps = NULL) is checked
against the Philox twin of test_gpu_noise.py, keyed on agent_base + g. In-kernel sampling writes its batch to `rows` and
its indices to `idx_out`: both must be bitwise the sampler twin's draw (oracle.philox_randint), and that batch is then the
reference's batch.

Ownership, as in test_gpu_row_kernels.run_wgrad: every output buffer starts as NaN inside a NaN guard band; every element
a kernel owns must come back finite and every other one must stay NaN (rows >= B, dZ3 columns past the head, slot 1 in an
actor step, LayerNorm partials without LayerNorm, the partial fields another kernel owns, the out fields, the gaps between
stacked agents). The arena, the counters and log alpha (critic / actor steps) and the rows (unless sampled in the kernel)
must be bitwise unchanged.

test_fused_bounds_have_teeth (no GPU) shows on small float64 references that each bound accepts an fp32 evaluation in
another order and rejects, at least tenfold, the mistakes these kernels can make.
"""
from __future__ import annotations

import ctypes as C
import math

import pytest
import torch

from tests.test_gpu_row_kernels import PART_DB3, PART_SCAL, PART_VEC, SHAPES, _bits, mean_ref, nblk_of, ws_carve, ws_floats
from tests.test_gpu_wide_kernels import (FLOOR, LOG_SQRT_2PI, LOG_STD_MAX, LOG_STD_MIN, ULP_EXP, ULP_LOG, ULP_TANH, WIDEN, WORST, R,
                                         U, _fp32_within, _lib, _teeth, check, f32, gam, group_sum, guarded, head_bwd_ref,
                                         policy_head_ref, q_target_ref, r_exp, r_sum, st, untouched)

HID, RT = 256, 8
INV_HID = 1.0 / HID  # (exact: a power of two)
LN_EPS = f32(1e-5)
SEED = 0x9E3779B97F4A7C15  # a Philox key with a non-zero high word
MASKS: dict = {}           # pass -> [units widened, units, kernel masks that differ from float64]


# ---- float64 references (plain torch; CPU or GPU) -------------------------------------------------------------------------
def rcat(*xs) -> R:
    xs = [R.of(x) for x in xs]
    return R(torch.cat([x.v for x in xs], 1), torch.cat([x.e for x in xs], 1))


def r_mm(x, w, b, k) -> R:
    """x [M][K] @ w [K][N] (+ b [N]): a sum whose longest chain is k roundings. x may carry its own bound (an R), which
    propagates through |w|."""
    x = R.of(x)
    w = w.double()
    aw = w.abs()
    v, s = x.v @ w, (x.v.abs() + x.e) @ aw
    if b is not None:
        v, s = v + b.double(), s + b.double().abs()
    return R(v, x.e @ aw + gam(k) * s)


def r_sqrt(a: R) -> R:
    v = torch.sqrt(a.v)
    return R(v, a.e / (v + torch.sqrt((a.v - a.e).clamp_min(0.0))) + U * v)


def layer_fwd(z: R, g, be, ln) -> dict:
    """layer_fwd_rows after row_stats: x-hat (or z), rstd, the pre-activation and h = ReLU of it."""
    if not ln:
        return dict(xh=z, rstd=None, pre=z, h=R(z.v.clamp_min(0.0), z.e))
    mean = r_sum(z, 1, 8) * INV_HID
    d = z - mean[:, None]
    rstd = R(1.0) / r_sqrt(r_sum(d * d, 1, 13) * INV_HID + LN_EPS)
    xh = d * rstd[:, None]
    pre = xh * g.double() + be.double()
    return dict(xh=xh, rstd=rstd, pre=pre, h=R(pre.v.clamp_min(0.0), pre.e))


def net_params(region, net) -> dict:
    """One net's tensors inside one arena region (fp32 views)."""
    t = lambda f, *s: None if net.off[f] < 0 else region[net.off[f]:net.off[f] + math.prod(s)].view(*s)
    p = {f: t(f, HID) for f in ("b1", "g1", "be1", "b2", "g2", "be2")}
    p.update(w1t=t("w1t", net.in_dim, HID), w2t=t("w2t", HID, HID), w3=t("w3", net.out_dim, HID), b3=t("b3", net.out_dim),
             ln=bool(net.layer_norm), in_dim=net.in_dim, out_dim=net.out_dim)
    return p


def trunk(X, p, h1=None) -> list:
    """Both hidden layers of one net on X [M][in_dim] (fp32, or an R). h1: the kernel's own first-layer activations, then
    the exact input of the second layer (each stored stage is checked from the kernel's stored input of that stage)."""
    l1 = layer_fwd(r_mm(X, p["w1t"], p["b1"], -(-p["in_dim"] // 8) + 8), p["g1"], p["be1"], p["ln"])
    l2 = layer_fwd(r_mm(l1["h"] if h1 is None else h1, p["w2t"], p["b2"], 40), p["g2"], p["be2"], p["ln"])
    return [l1, l2]


def head(layers, p) -> R:
    return r_mm(layers[1]["h"], p["w3"].T, p["b3"], 14)


def relu_mask(pre: R, what, h_kernel=None) -> R:
    """The backward pass's ReLU mask as an R (module docstring): the kernel's own (h_kernel > 0) where it stored the
    activations, else the float64 mask with R(0.5, 0.5) wherever |pre-activation| is within its bound."""
    near = pre.v.abs() <= WIDEN * pre.e + FLOOR
    stats = MASKS.setdefault(what, [0, 0, 0])
    stats[1] += near.numel()
    if h_kernel is not None:
        m = h_kernel > 0
        differ = m != (pre.v > 0)
        bad = differ & ~near
        assert not bool(bad.any()), (f"{what}: the kernel's ReLU mask differs from float64 away from a kink at (row, unit) "
                                     f"{bad.nonzero()[:4].tolist()}")
        stats[2] += int(differ.sum())
        return R(m.double(), torch.zeros_like(pre.v))
    stats[0] += int(near.sum())
    return R(torch.where(near, 0.5, (pre.v > 0).double()), torch.where(near, 0.5, 0.0))


def mask_mul(m: R, d) -> R:
    """m * d for a mask value in {0, 1} (exact) or R(0.5, 0.5) (either): no rounding."""
    d = R.of(d)
    return R(m.v * d.v, m.v * d.e + m.e * (d.v.abs() + d.e))


def layer_bwd(dh: R, layer, g, ln, m: R):
    """layer_bwd_rows: dz and the per-row terms of this layer's partials {b: dz, g: dn * x-hat, be: dn}."""
    dn = mask_mul(m, dh)
    if not ln:
        return dn, dict(b=dn)
    dx = dn * g.double()
    c1 = r_sum(dx, 1, 8) * INV_HID
    c2 = r_sum(dx * layer["xh"], 1, 8) * INV_HID
    dz = layer["rstd"][:, None] * ((dx - c1[:, None]) - layer["xh"] * c2[:, None])
    return dz, dict(b=dz, g=dn * layer["xh"], be=dn)


def trunk_bwd(dh2: R, layers, p, masks):
    """trunk_bwd: (dz1, dz2, [layer-1 terms, layer-2 terms]) from dLoss/dh2, masks [layer 1, layer 2]."""
    dz2, t2 = layer_bwd(dh2, layers[1], p["g2"], p["ln"], masks[1])
    dz1, t1 = layer_bwd(r_mm(dz2, p["w2t"].T, None, 39), layers[0], p["g1"], p["ln"], masks[0])
    return dz1, dz2, [t1, t2]


def tile_parts(terms) -> dict:
    """PART_VEC vectors per 8-row tile: {field index: R [nblk][256]}."""
    out = {}
    for layer, t in enumerate(terms):
        for i, f in enumerate(("b", "g", "be")):
            if f in t:
                out[3 * layer + i] = group_sum(t[f], RT, 7)
    return out


def next_action(pa, nobs, eps, lo, hi, td3, smoothing, std, c) -> dict:
    """The critic step's first pass on CTA 0: a' (and log pi) from next_obs; its layers kept for the sensitivity bound."""
    layers = trunk(nobs, pa)
    pol = policy_head_ref(None, None, None, eps, lo, hi, lo.shape[0], td3, smoothing, std, c, u=head(layers, pa))
    pol["layers"] = layers
    return pol


def q_pass(pq, X):
    layers = trunk(X, pq)
    return layers, head(layers, pq)[:, 0]


# ---- per-row scalars through passes that store nothing: a first-order bound by sensitivities --------------------------------
class Sens:
    """Adjoint running error analysis of a per-row scalar o. Every rounding adds a zero leaf d with its local bound (the R
    bound of that operation on exact operands); |error of o_r| <= sum over the leaves of row r of |d o_r / d leaf| * local
    (first order, widened like R), one backward pass for all rows (rows are independent). A bound carried forward |W|-wise
    through several 256-wide layers loses the weights' signs and grows ~sqrt(256) times per layer faster than this one. A unit
    within its R bound of a ReLU kink (of a clamp's edge, of a tie of min / max) passes no gradient and contributes |d o / d
    its output| times that R bound instead (a kink is 1-Lipschitz)."""

    def __init__(self):
        self.leaves = []

    def r(self, v, local):
        d = torch.zeros_like(v, requires_grad=True)
        self.leaves.append((d, torch.as_tensor(local, dtype=torch.float64, device=v.device).detach().expand_as(v)))
        return v + d

    def op(self, v, ulp_u=1):
        """one rounding: ulp_u u |v| (1 for the basic operations, 2 ulp per ulp of a transcendental)"""
        return self.r(v, ulp_u * U * v.detach().abs())

    def kink(self, v, near, e):
        """v (in the graph) where no unit is near a kink; near ones pass no gradient and add their bound e"""
        return self.r(torch.where(near, v.detach(), v), torch.where(near, e, 0.0))

    def dot(self, x, w, b, k):
        w = w.double()
        v, s = x @ w, x.detach().abs() @ w.abs()
        if b is not None:
            v, s = v + b.double(), s + b.double().abs()
        return self.r(v, gam(k) * s)

    def bound(self, o):
        gs = torch.autograd.grad(o.sum(), [d for d, _ in self.leaves], allow_unused=True, retain_graph=True)
        e = torch.zeros_like(o.detach())
        for (_, loc), g in zip(self.leaves, gs):
            if g is not None:
                e = e + (g.abs() * loc).reshape(o.shape[0], -1).sum(1)
        return e


def s_trunk(S, X, p, rl):
    """trunk (head included) in the Sens form; rl: the R form's layers of the same pass (their kink bounds)."""
    h = X
    for i, k in enumerate((-(-p["in_dim"] // 8) + 8, 40)):
        n = str(i + 1)
        z = S.dot(h, p["w" + n + "t"], p["b" + n], k)
        if p["ln"]:
            mean = S.r(z.sum(1, keepdim=True) * INV_HID, gam(8) * z.detach().abs().sum(1, keepdim=True) * INV_HID)
            d = S.op(z - mean)
            var = S.r((d * d).sum(1, keepdim=True) * INV_HID, gam(13) * (d.detach() ** 2).sum(1, keepdim=True) * INV_HID)
            rstd = S.op(1.0 / S.op(torch.sqrt(S.op(var + LN_EPS))))
            pre = S.op(S.op(d * rstd) * p["g" + n].double() + p["be" + n].double())
        else:
            pre = z
        rp = rl[i]["pre"]
        h = S.kink(pre.clamp_min(0.0), rp.v.abs() <= WIDEN * rp.e + FLOOR, rp.e)
    return S.dot(h, p["w3"].T, p["b3"], 14)


def s_policy(S, u, eps, lo, hi, td3, smoothing, std, c, rpol):
    """policy.cuh in the Sens form: (action, log pi or None)."""
    B, A = u.shape[0], lo.shape[0]
    lo64, hi64 = lo.double().expand(B, A), hi.double().expand(B, A)
    scale, bias = S.op(hi64 - lo64) * 0.5, S.op(hi64 + lo64) * 0.5
    eps = eps.double()
    if td3:
        act = S.op(S.op(S.op(torch.tanh(u[:, :A]), 2 * ULP_TANH) * scale) + bias)
        if not smoothing:
            return act, None
        n = S.op(eps * f32(std))
        cc = f32(c)
        n = S.kink(n.clamp(-cc, cc), (n.detach().abs() - cc).abs() <= U * n.detach().abs() + FLOOR, U * n.detach().abs())
        s = S.op(act + n)
        e = rpol["act"].e
        near = ((s.detach() - lo64).abs() <= WIDEN * e + FLOOR) | ((s.detach() - hi64).abs() <= WIDEN * e + FLOOR)
        return S.kink(torch.minimum(torch.maximum(s, lo64), hi64), near, e), None
    mu, raw = u[:, :A], u[:, A:2 * A]
    th = S.op(torch.tanh(raw), 2 * ULP_TANH)
    ls = S.op(LOG_STD_MIN + S.op((0.5 * (LOG_STD_MAX - LOG_STD_MIN)) * S.op(th + 1.0)))
    sigma = S.op(torch.exp(ls), 2 * ULP_EXP)
    x = S.op(mu + S.op(eps * sigma))
    y = S.op(torch.tanh(x), 2 * ULP_TANH)
    act = S.op(S.op(y * scale) + bias)
    d = S.op(x - mu)
    logn = S.op(S.op(-S.op(S.op(d * d) / (2.0 * S.op(sigma * sigma))) - S.op(torch.log(sigma), 2 * ULP_LOG)) - LOG_SQRT_2PI)
    corr = S.op(torch.log(S.op(S.op(scale * S.op(1.0 - S.op(y * y))) + f32(1e-6))), 2 * ULP_LOG)
    lp = S.op(logn - corr)
    return act, S.r(lp.sum(1), gam(max(A - 1, 1)) * lp.detach().abs().sum(1))


def y_sens_bound(P, T, lay, batch, eps, lo, hi, log_alpha, gamma, std, c, td3, bcq, smoothing, rpol, rqn):
    """The Sens bound of the TD target y (the next-action pass, both target passes, min / BCQ mix, the entropy term)."""
    obs, act, rew, done, nobs = batch
    S = Sens()
    with torch.enable_grad():
        pa = net_params(T if td3 else P, lay.actor)
        a2, logp = s_policy(S, s_trunk(S, nobs.double(), pa, rpol["layers"]), eps, lo, hi, td3, smoothing, std, c, rpol)
        X = torch.cat([nobs.double(), a2], 1)
        qn = [s_trunk(S, X, net_params(T, lay.critic[k]), rqn[k][0])[:, 0] for k in range(2)]
        e_q = torch.maximum(rqn[0][1].e, rqn[1][1].e)
        tie = (qn[0] - qn[1]).detach().abs() <= WIDEN * (rqn[0][1].e + rqn[1][1].e) + FLOOR
        qp = S.kink(torch.minimum(*qn), tie, e_q)
        if bcq:
            qp = S.op(S.op(0.75 * qp) + S.op(0.25 * S.kink(torch.maximum(*qn), tie, e_q)))
        if not td3:
            alpha = S.op(torch.exp(log_alpha.double()).expand_as(qp), 2 * ULP_EXP)
            qp = S.op(qp - S.op(alpha * logp))
        y = S.op(rew.double() + S.op(S.op((1.0 - done.double()) * f32(gamma)) * qp))
        return S.bound(y)


def tighten_policy(pa, X, eps, lo, hi, td3, smoothing, std, c, rpol):
    """rpol (policy_head_ref's R values of a pass on X) with the bounds of the action and log pi replaced by the smaller of
    their R and Sens bounds (one backward pass per action dimension): the passes that take the action as input then start
    from a tight bound, and so do their kink tests."""
    S = Sens()
    with torch.enable_grad():
        act, logp = s_policy(S, s_trunk(S, X.double(), pa, rpol["layers"]), eps, lo, hi, td3, smoothing, std, c, rpol)
        ea = torch.stack([S.bound(act[:, i]) for i in range(act.shape[1])], 1)
        rpol["act"] = R(rpol["act"].v, torch.fmin(rpol["act"].e, ea))
        if logp is not None:
            rpol["logp"] = R(rpol["logp"].v, torch.fmin(rpol["logp"].e, S.bound(logp)))
    return rpol


# ---- the three kernels' references ------------------------------------------------------------------------------------------
def critic_step_ref(P, T, lay, batch, eps, lo, hi, log_alpha, gamma, std, c, td3, bcq, smoothing, kern):
    """critic_fused for one agent. The TD target from scratch (its passes store nothing: the smaller of its R and Sens
    bounds); every stored stage from the kernel's own stored input of that stage — kern["y"], and per critic k kern["k"][k]
    = the workspace h1, h2, dz1, dz2, dZ3 column 0 of slot k and Q — which keeps each bound tight and checks every stage."""
    obs, act, rew, done, nobs = batch
    B = obs.shape[0]
    pa = net_params(T if td3 else P, lay.actor)
    pol = tighten_policy(pa, nobs, eps, lo, hi, td3, smoothing, std, c, next_action(pa, nobs, eps, lo, hi, td3, smoothing, std, c))
    Xn = rcat(nobs, pol["act"])
    qn = [q_pass(net_params(T, lay.critic[k]), Xn) for k in range(2)]
    y = q_target_ref(qn[0][1], qn[0][1], qn[1][1], pol.get("logp"), log_alpha, rew, done, gamma, B, td3, bcq)["y"]
    e_s = y_sens_bound(P, T, lay, batch, eps, lo, hi, log_alpha, gamma, std, c, td3, bcq, smoothing, pol, qn)
    out = dict(y=R(y.v, torch.fmin(y.e, e_s)), sat=None if td3 else pol["sat"].any(1), k=[], pol=pol, qn=qn)
    X = torch.cat([obs, act], 1)
    two_b = R(2.0) / R(float(B))
    for k in range(2):
        kk = kern["k"][k]
        po = net_params(P, lay.critic[k])
        layers = trunk(X, po, h1=kk["h1"])
        dlt = R(kk["q"]) - R(kern["y"])
        masks = [relu_mask(layers[i]["pre"], f"critic step, online critic, layer {i + 1}", kk["h" + str(i + 1)]) for i in range(2)]
        dz2, t2 = layer_bwd(R(kk["dz3"])[:, None] * po["w3"][0], layers[1], po["g2"], po["ln"], masks[1])
        dz1, t1 = layer_bwd(r_mm(kk["dz2"], po["w2t"].T, None, 39), layers[0], po["g1"], po["ln"], masks[0])
        t1["b"], t2["b"] = R(kk["dz1"]), R(kk["dz2"])  # (each tile sums the kernel's own dz)
        out["k"].append(dict(q=r_mm(kk["h2"], po["w3"].T, po["b3"], 14)[:, 0], h1=layers[0]["h"], h2=layers[1]["h"], layers=layers,
                             dz=dlt * two_b, dz1=dz1, dz2=dz2, parts=tile_parts([t1, t2]), db3=group_sum(R(kk["dz3"])[:, None], RT, 7)[:, 0],
                             sq=group_sum((dlt * dlt)[:, None], RT, 7)[:, 0]))
    return out


def actor_step_ref(P, lay, obs, eps, lo, hi, log_alpha, td3, kern, c_pi_rows=None):
    """actor_fused for one agent: the actor's activations, dZ3 [B][out_dim] (g_mu | g_raw, or g_a), dZ1 / dZ2 and the tile
    partials (vectors, head bias, loss, log pi). kern: the workspace h1, h2, dz1, dz2 and dZ3 [:, :out_dim] of slot 0, each
    stored stage's exact input. The critic passes store nothing: their bounds are the R form's, with the widened masks.
    c_pi_rows: the M of c_pi = alpha * fl(1 / M) (B; a mistake for the teeth test)."""
    B, O, A = obs.shape[0], obs.shape[1], lo.shape[0]
    pa = net_params(P, lay.actor)
    la = trunk(obs, pa, h1=kern["h1"])
    pol = policy_head_ref(None, None, None, eps, lo, hi, A, td3, u=r_mm(kern["h2"], pa["w3"].T, pa["b3"], 14))
    X = rcat(obs, pol["act"])
    inv_b = R(1.0) / R(float(B))
    ks = (0,) if td3 else (0, 1)
    qs = [q_pass(net_params(P, lay.critic[k]), X) for k in ks]
    if td3:
        choice = [R(torch.ones_like(qs[0][1].v))]
        loss = -qs[0][1]
        lp = R(torch.zeros_like(loss.v))
    else:
        (_, q0), (_, q1) = qs
        first = q0.v <= q1.v
        near = (q0.v - q1.v).abs() <= WIDEN * (q0.e + q1.e) + FLOOR
        st_ = MASKS.setdefault("actor step, arg-min of Q0, Q1", [0, 0, 0])
        st_[0] += int(near.sum())
        st_[1] += near.numel()
        c0 = R(torch.where(near, 0.5, first.double()), torch.where(near, 0.5, 0.0))
        choice = [c0, R(1.0 - c0.v, c0.e)]
        qsel = R(torch.where(first, q0.v, q1.v), torch.maximum(q0.e, q1.e) + torch.where(near, (q0.v - q1.v).abs(), 0.0))
        loss = r_exp(R(log_alpha)) * pol["logp"] - qsel
        lp = pol["logp"]
    da = []
    for (layers, _), k, ch in zip(qs, ks, choice):
        pq = net_params(P, lay.critic[k])
        masks = [relu_mask(layers[i]["pre"], f"actor step, critic, layer {i + 1}") for i in range(2)]
        dz1, _, _ = trunk_bwd(mask_mul(ch, -inv_b)[:, None] * pq["w3"][0], layers, pq, masks)
        da.append(r_mm(dz1, pq["w1t"][O:O + A].T, None, 13))
    save = [None, None, None, pol["th"]] if td3 else [pol["eps"], pol["sigma"], pol["y"], pol["th"]]
    hb = head_bwd_ref(da[0], None if td3 else da[1], save, lo, hi, log_alpha, td3, A, c_pi_rows or B, recip=True)
    masks = [relu_mask(la[i]["pre"], f"actor step, actor, layer {i + 1}", kern["h" + str(i + 1)]) for i in range(2)]
    dz2, t2 = layer_bwd(r_mm(kern["dz3"], pa["w3"], None, pa["out_dim"]), la[1], pa["g2"], pa["ln"], masks[1])
    dz1, t1 = layer_bwd(r_mm(kern["dz2"], pa["w2t"].T, None, 39), la[0], pa["g1"], pa["ln"], masks[0])
    t1["b"], t2["b"] = R(kern["dz1"]), R(kern["dz2"])
    return dict(h1=la[0]["h"], h2=la[1]["h"], du=hb["du"], du_sat=hb["sat"], dz1=dz1, dz2=dz2, parts=tile_parts([t1, t2]),
                db3=group_sum(R(kern["dz3"]), RT, 3), loss=group_sum(loss[:, None], RT, 7)[:, 0], lp=group_sum(lp[:, None], RT, 7)[:, 0],
                sat=None if td3 else pol["sat"].any(1), da=da, layers=la, pol=pol)


def alpha_terms_ref(P, lay, obs, eps2, lo, hi, targ_ent) -> dict:
    """alpha_kernel's rows: -log pi - targ_ent of a fresh sample of the actor (log pi under the smaller of its R and Sens
    bounds), and their 8-row tile sums."""
    pa = net_params(P, lay.actor)
    layers = trunk(obs, pa)
    pol = policy_head_ref(None, None, None, eps2, lo, hi, lo.shape[0], False, u=head(layers, pa))
    pol["layers"] = layers
    t = (-tighten_policy(pa, obs, eps2, lo, hi, False, False, 0.0, 0.0, pol)["logp"]) - f32(targ_ent)
    return dict(t=t, part=group_sum(t[:, None], RT, 7)[:, 0], sat=pol["sat"].any(1))


# ---- inputs -----------------------------------------------------------------------------------------------------------------
def _opts(s: str) -> dict:
    o = set(filter(None, s.split(",")))
    return dict(ln=None if not ({"ln0", "ln1"} & o) else "ln1" in o, bcq="bcq" in o, smoothing="smooth0" not in o,
                autotune="auto0" not in o, sym="sym" in o, table="table" in o, dev_noise="dev" in o, sample="sample" in o)


def _fill_region(reg, lay, g, shift=None):
    """Parameters of the three nets in one region (the padding between tensors stays NaN); shift: a region to perturb."""
    for net in (*lay.critic, lay.actor):
        def put(f, v):
            o = net.off[f]
            reg[o:o + net.numel(f)] = v.reshape(-1) if shift is None else shift[o:o + net.numel(f)] + 0.2 * v.reshape(-1)
        rn = lambda *s: torch.randn(*s, device="cuda", generator=g)
        put("w1t", rn(net.in_dim, HID) * (1.5 / math.sqrt(net.in_dim)))
        put("b1", 0.2 * rn(HID))
        put("w2t", rn(HID, HID) / 12.0)
        put("b2", 0.2 * rn(HID))
        if net.layer_norm:
            for f in ("g1", "g2"):
                put(f, 1.0 + 0.2 * rn(HID) if shift is None else 0.2 * rn(HID))
            for f in ("be1", "be2"):
                put(f, 0.2 * rn(HID))
        put("w3", rn(net.out_dim, HID) / 12.0)
        put("b3", 0.3 * rn(net.out_dim))
        o, w = net.off["w2n"], net.off["w2t"]
        reg[o:o + HID * HID] = reg[w:w + HID * HID].view(HID, HID).t().reshape(-1)


def _table(td3, n, A):
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.population import agent_hp_table, agent_hp_values
    hps = (td3_hps if td3 else sac_hps)(batch_size=256)
    over = dict(gamma=[0.99, 0.9, 0.5][:n], targ_ent=[-3.0, -1.5, 0.25][:n], log_alpha_lr=[3e-4, 1e-2, 0.05][:n])
    if td3:
        over.update(td3_std=[0.3, 0.6, 0.1][:n], td3_c=[0.5, 0.25, 0.05][:n])
    vals = agent_hp_values(hps, n, A, over)
    return torch.from_numpy(agent_hp_table(vals, td3)).cuda(), vals


def run_case(L, shape, B, n, opts, which, seed=0):
    """Inputs of one case and one b2rl_launch_single launch of kernel `which` (0 critic_fused, 2 actor_fused, 4 alpha)."""
    from sac_td3_cudagraphs_pytorch_b200.arena import _up4, make_layout
    lib = L.load()
    ob, ac, td3, ln = SHAPES[shape]
    o = _opts(opts)
    ln = ln if o["ln"] is None else o["ln"]
    lay = make_layout(ob, ac, td3, ln)
    rs = _up4(2 * ob + ac + 2)
    g = torch.Generator(device="cuda").manual_seed(seed + 131 * B + 17 * n + 1000 * len(opts) + 7 * ob + ac)
    rn = lambda *s: torch.randn(*s, device="cuda", generator=g)
    gap = 12 if n > 1 else 0
    base = 5 if n > 1 else 0
    ars, rws = 5 * lay.region + gap, B * rs + gap
    wsf = ws_floats(B)
    assert wsf == lib.b2rl_workspace_floats(B)
    wss = wsf + gap
    ar_f, ar = guarded(n, ars)
    for a in range(n):
        _fill_region(ar[a, :lay.region], lay, g)
        _fill_region(ar[a, lay.region:2 * lay.region], lay, g, shift=ar[a, :lay.region].clone())  # the target nets
    if o["sym"]:
        lo, hi = -torch.ones(ac, device="cuda"), torch.ones(ac, device="cuda")
    else:
        lo = -0.5 - torch.rand(ac, device="cuda", generator=g)
        hi = 0.2 + 1.5 * torch.rand(ac, device="cuda", generator=g)
    rw_f, rw = guarded(n, rws)
    for a in range(n):
        rows = rw[a, :B * rs].view(B, rs)
        rows[:, :ob] = 1.5 * rn(B, ob)
        rows[:, ob:ob + ac] = lo + (hi - lo) * torch.rand(B, ac, device="cuda", generator=g)
        rows[:, ob + ac] = rn(B)
        rows[:, ob + ac + 1] = (torch.rand(B, device="cuda", generator=g) < 0.3).float()
        rows[:, ob + ac + 2:2 * ob + ac + 2] = 1.5 * rn(B, ob)  # (the padding columns stay NaN)
    ws_f, ws = guarded(n, wss)
    la_f, la = guarded(n, 5)
    la[:, 0] = torch.tensor([-1.3, 0.4, -0.2][:n], device="cuda")
    la[:, 2] = 0.01 * rn(n)
    la[:, 3] = 1e-4 * torch.rand(n, device="cuda", generator=g)
    o_f, out = guarded(n, 8)
    ctr = torch.zeros(n, 8, dtype=torch.int64, device="cuda")
    ctr[:, L.CTR_Q] = torch.arange(n, device="cuda") + 11
    ctr[:, L.CTR_PI] = torch.arange(n, device="cuda") + 23
    ctr[:, L.CTR_ALPHA] = torch.arange(n, device="cuda") + 4
    eps = None if o["dev_noise"] else rn(n, B, ac)
    eo_f, eo = guarded(n, B, ac)
    tq_f, tq = guarded(n, B)
    q_f, qv = guarded(n, 2, B)
    hp, vals = _table(td3, n, ac) if o["table"] else (None, None)
    a = L.UpdateArgs()
    a.hp = L.Hyper(td3=int(td3), bcq_mix=int(o["bcq"]), targ_smoothing=int(o["smoothing"]), autotune=int(o["autotune"]), gamma=0.97,
                   td3_std=0.2, td3_c=0.5, targ_ent=-float(ac), seed=SEED)
    a.fmt = L.RowFmt(ob, ac, rs, 0)
    a.actor = lay.actor.c_struct()
    a.critic[0], a.critic[1] = lay.critic[0].c_struct(), lay.critic[1].c_struct()
    a.batch, a.n_agents, a.agent_base = B, n, base
    a.region_stride, a.arena_agent_stride = lay.region, ars
    a.arena, a.rows, a.rows_agent_stride = ar.data_ptr(), rw.data_ptr(), rws
    a.min_ac, a.max_ac, a.log_alpha, a.counters = lo.data_ptr(), hi.data_ptr(), la.data_ptr(), ctr.data_ptr()
    a.workspace, a.workspace_agent_stride, a.out = ws.data_ptr(), wss, out.data_ptr()
    if which == 4:
        a.eps2, a.eps2_out = None if eps is None else eps.data_ptr(), eo.data_ptr()
    else:
        a.eps, a.eps_out = None if eps is None else eps.data_ptr(), eo.data_ptr()
    a.dbg_targ_q, a.dbg_q = tq.data_ptr(), qv.data_ptr()
    a.agent_hp = None if hp is None else hp.data_ptr()
    smp = None
    if o["sample"]:  # 95 of 100 replay rows filled, 10 new rows appended at cursor 95 (they wrap to rows 0-4)
        assert n == 1 and which == 0
        cap, n_new, cursor = 100, 10, 95
        sto = rn(cap, rs)
        sto[:, ob + ac + 1] = (torch.rand(cap, device="cuda", generator=g) < 0.3).float()
        new = rn(n_new, rs)
        new[:, ob + ac + 1] = 1.0
        ctr[:, L.CTR_SIZE], ctr[:, L.CTR_CURSOR] = cap - 5, cursor
        idx = torch.full((n, B), -1, dtype=torch.int64, device="cuda")
        a.storage, a.storage_agent_stride, a.storage_size = sto.data_ptr(), cap * rs, 0
        a.idx_out, a.new_rows, a.capacity, a.n_new = idx.data_ptr(), new.data_ptr(), cap, n_new
        smp = dict(sto=sto, new=new, idx=idx, cap=cap, n_new=n_new, cursor=cursor, size=min(cap - 5 + n_new, cap))
    before = dict(ar=_bits(ar_f), rw=_bits(rw_f), la=_bits(la_f), la_v=la.clone(), ctr=ctr.clone())
    L.check(lib.b2rl_launch_single(C.byref(a), which, st()), f"launch_single {which}")
    torch.cuda.synchronize()
    gam_ = [f32(v["gamma"]) for v in vals] if vals else [f32(0.97)] * n
    std_ = [f32(v["td3_std"]) for v in vals] if (vals and td3) else [f32(0.2)] * n
    c_ = [f32(v["td3_c"]) for v in vals] if (vals and td3) else [f32(0.5)] * n
    te_ = [f32(v["targ_ent"]) for v in vals] if vals else [f32(-float(ac))] * n
    lr_ = [f32(v["log_alpha_lr"]) for v in vals] if vals else [f32(1e-3)] * n
    return dict(lay=lay, ob=ob, ac=ac, td3=td3, ln=ln, o=o, rs=rs, B=B, n=n, base=base, ar_f=ar_f, ar=ar, rw_f=rw_f, rw=rw, ws_f=ws_f,
                ws=ws, la_f=la_f, la=la, o_f=o_f, out=out, ctr=ctr, eps=eps, eo_f=eo_f, eo=eo, tq_f=tq_f, tq=tq, q_f=q_f, qv=qv,
                lo=lo, hi=hi, before=before, gamma=gam_, std=std_, c=c_, te=te_, lr=lr_, smp=smp,
                tag=f"{shape} B={B} n={n} {opts or 'default'}")


def _batch(r, a):
    ob, ac, B = r["ob"], r["ac"], r["B"]
    rows = r["rw"][a, :B * r["rs"]].view(B, r["rs"])
    return rows[:, :ob], rows[:, ob:ob + ac], rows[:, ob + ac], rows[:, ob + ac + 1], rows[:, ob + ac + 2:2 * ob + ac + 2]


def _check_noise(r, a, stream, step_ctr, used):
    """eps_out: the given noise bitwise, or the Philox twin's draw keyed on agent_base + a; untouched when not drawn."""
    from tests.test_gpu_noise import check_noise
    got = r["eo"][a]
    if not used:
        assert torch.isnan(got).all(), r["tag"] + ": eps_out written, but no noise is drawn"
        return None
    if r["eps"] is not None:
        assert torch.equal(_bits(got), _bits(r["eps"][a])), r["tag"] + ": eps_out is not the given noise"
    else:
        check_noise(f"{r['tag']} agent {a} noise", got, SEED, int(r["before"]["ctr"][a, step_ctr]), stream, r["base"] + a)
    return got


def _part_own(own_part, ln, extra):
    for v in (range(PART_VEC) if ln else (0, 3)):
        own_part[:, v * HID:(v + 1) * HID] = True
    for i in extra:
        own_part[:, i] = True


def _check_parts(kind, tag, part, ref_parts):
    for v, ref in ref_parts.items():
        check(kind, f"{tag} part vector {v}", part[:, v * HID:(v + 1) * HID], ref)


def _common_untouched(r, ws_own, what):
    untouched(r["ws_f"], r["ws"], ~ws_own, f"{what}: workspace")
    assert torch.equal(_bits(r["ar_f"]), r["before"]["ar"]), f"{what}: the arena changed"


# ---- critic_fused ------------------------------------------------------------------------------------------------------------
HOPPER_B = (1, 7, 8, 9, 255, 256, 257, 263, 4097, 65536, 65543)
FUSED_CASES = (
    [(s, B, 1, "") for s in ("hopper_sac", "hopper_td3") for B in HOPPER_B]
    + [("humanoid_sac", B, 1, "") for B in (7, 257, 4097)]
    + [("one_one", B, 1, "") for B in (1, 9, 263)]
    + [("in31_32", B, 1, "") for B in (8, 257)]
    + [("in32_33", B, 1, "") for B in (9, 263)]
    + [("a32_sac", B, 1, "") for B in (255, 4097)]
    # LayerNorm on / off against the shape's default, BCQ mix, no target smoothing, symmetric bounds, no autotune
    + [("hopper_sac", 263, 1, "ln0,bcq"), ("hopper_sac", 257, 1, "sym,auto0"), ("hopper_td3", 263, 1, "ln1,bcq"),
       ("hopper_td3", 257, 1, "smooth0"), ("hopper_td3", 9, 1, "sym,bcq"), ("humanoid_sac", 9, 1, "ln0,bcq"),
       ("in31_32", 263, 1, "ln0,smooth0"), ("in32_33", 257, 1, "ln1,bcq"), ("a32_sac", 9, 1, "ln0,sym")]
    # stacked agents (agent_base 5, NaN gaps), with and without a per-agent table
    + [("hopper_sac", 1000, 3, "table"), ("hopper_td3", 263, 3, "table,bcq"), ("hopper_sac", 257, 3, "")]
    # device-drawn noise
    + [("hopper_sac", 263, 3, "dev,table"), ("hopper_td3", 257, 1, "dev"), ("humanoid_sac", 9, 1, "dev")]
    # in-kernel sampling with new rows that wrap the cursor
    + [("hopper_sac", 263, 1, "sample"), ("hopper_td3", 257, 1, "sample,dev")]
)


def check_critic(L, r):
    lay, B, n, ob, ac, td3, o = r["lay"], r["B"], r["n"], r["ob"], r["ac"], r["td3"], r["o"]
    ws_own = torch.zeros_like(r["ws"], dtype=torch.bool)
    for a in range(n):
        tag = f"{r['tag']} agent {a}"
        if r["smp"] is not None:  # the batch the kernel drew and wrote back, against the sampler twin
            from oracle import philox_randint
            s = r["smp"]
            want = torch.from_numpy(philox_randint(SEED, int(r["before"]["ctr"][a, L.CTR_Q]), s["size"], B, r["base"] + a)).cuda()
            assert torch.equal(s["idx"][a], want), tag + ": idx_out is not the sampler twin's draw"
            j = (want - s["cursor"]) % s["cap"]
            rows = torch.where((j < s["n_new"])[:, None], s["new"][j.clamp_max(s["n_new"] - 1)], s["sto"][want])
            assert torch.equal(_bits(r["rw"][a, :B * r["rs"]].view(B, r["rs"])), _bits(rows)), tag + ": sampled rows differ from the twin's"
        obs, act, rew, done, nobs = _batch(r, a)
        noise = _check_noise(r, a, 1, L.CTR_Q, not td3 or o["smoothing"])
        eps = noise if noise is not None else torch.zeros(B, ac, device="cuda")
        kern = dict(y=r["tq"][a], k=[])
        for k in range(2):
            w = ws_carve(r["ws"][a], B, k)
            kern["k"].append(dict(h1=w["h1"], h2=w["h2"], dz1=w["dz1"], dz2=w["dz2"], dz3=w["dz3"][:, 0], q=r["qv"][a, k]))
            for f, v in kern["k"][k].items():
                assert torch.isfinite(v).all(), f"{tag}: {f} of critic {k} not written (or not finite)"
        assert torch.isfinite(kern["y"]).all(), f"{tag}: y not written (or not finite)"
        P, T = r["ar"][a, :lay.region], r["ar"][a, lay.region:2 * lay.region]
        ref = critic_step_ref(P, T, lay, (obs, act, rew, done, nobs), eps, r["lo"], r["hi"], r["la"][a, 0].double(), r["gamma"][a],
                              r["std"][a], r["c"][a], td3, o["bcq"], o["smoothing"], kern)
        check("fused critic y", tag, r["tq"][a], ref["y"], ref["sat"])
        for k in range(2):
            t, rk = f"{tag} critic {k}", ref["k"][k]
            w = ws_carve(r["ws"][a], B, k)
            check("fused critic Q", t, r["qv"][a, k], rk["q"])
            check("fused critic h", t + " h1", w["h1"], rk["h1"])
            check("fused critic h", t + " h2", w["h2"], rk["h2"])
            check("fused critic dz3", t, w["dz3"][:, 0], rk["dz"])
            check("fused critic dz", t + " dz2", w["dz2"], rk["dz2"])
            check("fused critic dz", t + " dz1", w["dz1"], rk["dz1"])
            _check_parts("fused critic part", t, w["part"], rk["parts"])
            check("fused critic part scalars", t + " db3", w["part"][:, PART_DB3], rk["db3"])
            check("fused critic part scalars", t + " sum sq", w["part"][:, PART_SCAL], rk["sq"])
            wo = ws_carve(ws_own[a], B, k)
            for f in ("h1", "h2", "dz1", "dz2"):
                wo[f][:] = True
            wo["dz3"][:, 0] = True
            _part_own(wo["part"], r["ln"], (PART_DB3, PART_SCAL))
    _common_untouched(r, ws_own, r["tag"])
    untouched(r["tq_f"], what="dbg_targ_q")
    untouched(r["q_f"], what="dbg_q")
    untouched(r["eo_f"], what="eps_out")
    untouched(r["o_f"], r["out"], torch.ones_like(r["out"], dtype=torch.bool), "out (critic_fused writes none)")
    assert torch.equal(_bits(r["la_f"]), r["before"]["la"]), "log alpha changed"
    assert torch.equal(r["ctr"], r["before"]["ctr"]), "critic_fused bumped a counter"
    if r["smp"] is None:
        assert torch.equal(_bits(r["rw_f"]), r["before"]["rw"]), "the rows changed"
    else:
        assert torch.isnan(r["rw_f"][:64]).all() and torch.isnan(r["rw_f"][-64:]).all(), "rows: written outside the buffer"


@pytest.mark.gpu
@pytest.mark.parametrize("shape,B,n,opts", FUSED_CASES)
def test_critic_fused_matches_float64(shape, B, n, opts):
    """critic_fused alone: the TD target, both critics' Q, the workspace activations and gradients of both slots, dZ3
    column 0 and every tile's partials, each row against float64; the noise, the sampled batch and ownership."""
    L = _lib()
    check_critic(L, run_case(L, shape, B, n, opts, 0))


# ---- actor_fused -------------------------------------------------------------------------------------------------------------
def check_actor(L, r):
    lay, B, n, td3, o = r["lay"], r["B"], r["n"], r["td3"], r["o"]
    od = lay.actor.out_dim
    ws_own = torch.zeros_like(r["ws"], dtype=torch.bool)
    for a in range(n):
        tag = f"{r['tag']} agent {a}"
        obs = _batch(r, a)[0]
        noise = _check_noise(r, a, 2, L.CTR_PI, not td3)
        w = ws_carve(r["ws"][a], B, 0)
        kern = dict(h1=w["h1"], h2=w["h2"], dz1=w["dz1"], dz2=w["dz2"], dz3=w["dz3"][:, :od])
        for f, v in kern.items():
            assert torch.isfinite(v).all(), f"{tag}: actor {f} not written (or not finite)"
        ref = actor_step_ref(r["ar"][a, :lay.region], lay, obs, noise if noise is not None else torch.zeros(B, r["ac"], device="cuda"),
                             r["lo"], r["hi"], r["la"][a, 0].double(), td3, kern)
        sat = ref["sat"]
        check("fused actor h", tag + " h1", w["h1"], ref["h1"])
        check("fused actor h", tag + " h2", w["h2"], ref["h2"])
        check("fused actor dz3", tag, w["dz3"][:, :od], ref["du"], ref["du_sat"])
        check("fused actor dz", tag + " dz2", w["dz2"], ref["dz2"])
        check("fused actor dz", tag + " dz1", w["dz1"], ref["dz1"])
        _check_parts("fused actor part", tag, w["part"], ref["parts"])
        tile_sat = None if sat is None else group_sum(R(sat[:, None].double()), RT, 0).v[:, 0] > 0
        check("fused actor part scalars", tag + " db3", w["part"][:, PART_DB3:PART_DB3 + od], ref["db3"])
        check("fused actor part scalars", tag + " loss", w["part"][:, PART_SCAL], ref["loss"], tile_sat)
        check("fused actor part scalars", tag + " log pi", w["part"][:, PART_SCAL + 1], ref["lp"], tile_sat)
        wo = ws_carve(ws_own[a], B, 0)
        for f in ("h1", "h2", "dz1", "dz2"):
            wo[f][:] = True
        wo["dz3"][:, :od] = True
        _part_own(wo["part"], r["ln"], list(range(PART_DB3, PART_DB3 + od)) + [PART_SCAL, PART_SCAL + 1])
    _common_untouched(r, ws_own, r["tag"])
    untouched(r["eo_f"], what="eps_out")
    untouched(r["o_f"], r["out"], torch.ones_like(r["out"], dtype=torch.bool), "out (actor_fused writes none)")
    untouched(r["tq_f"], r["tq"], torch.ones_like(r["tq"], dtype=torch.bool), "dbg_targ_q")
    untouched(r["q_f"], r["qv"], torch.ones_like(r["qv"], dtype=torch.bool), "dbg_q")
    assert torch.equal(_bits(r["la_f"]), r["before"]["la"]), "log alpha changed"
    assert torch.equal(r["ctr"], r["before"]["ctr"]), "actor_fused bumped a counter"
    assert torch.equal(_bits(r["rw_f"]), r["before"]["rw"]), "the rows changed"


ACTOR_CASES = [c for c in FUSED_CASES if "sample" not in c[3]]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,B,n,opts", ACTOR_CASES)
def test_actor_fused_matches_float64(shape, B, n, opts):
    """actor_fused alone: the actor's activations and gradients (workspace slot 0), dZ3 (g_mu | g_raw, or g_a), every
    tile's partials with the loss and log pi sums, each row against float64, through both critics' backward passes with
    the interval masks; the noise and ownership (slot 1 stays NaN)."""
    L = _lib()
    check_actor(L, run_case(L, shape, B, n, opts, 2))


# ---- alpha_kernel ------------------------------------------------------------------------------------------------------------
def check_alpha(L, r):
    from tests.test_gpu_optimizer import EXP_ULP, adam_bound, adam_ref
    lay, B, n = r["lay"], r["B"], r["n"]
    ws_own = torch.zeros_like(r["ws"], dtype=torch.bool)
    o_own = torch.zeros_like(r["out"], dtype=torch.bool)
    la0 = r["before"]["la_v"].view(-1).cpu().double().numpy()
    for a in range(n):
        tag = f"{r['tag']} agent {a}"
        obs = _batch(r, a)[0]
        noise = _check_noise(r, a, 3, L.CTR_PI, True)
        ref = alpha_terms_ref(r["ar"][a, :lay.region], lay, obs, noise, r["lo"], r["hi"], r["te"][a])
        part = ws_carve(r["ws"][a], B, 0)["part"][:, PART_SCAL + 2]
        tile_sat = group_sum(R(ref["sat"][:, None].double()), RT, 0).v[:, 0] > 0
        check("fused alpha partials", tag, part, ref["part"], tile_sat)
        ws_carve(ws_own[a], B, 0)["part"][:, PART_SCAL + 2] = True
        # the last cluster: alpha * mean of the kernel's own partials, then one Adam step of log alpha
        loss = r_exp(R(torch.tensor(la0[a * 5], dtype=torch.float64))) * mean_ref(part.double().cpu(), B)
        check("fused alpha loss", tag, r["out"][a, L.OUT_ALPHA_LOSS].cpu(), loss)
        g = float(r["out"][a, L.OUT_ALPHA_LOSS])
        assert r["la"][a, 1].item() == g, tag + ": log alpha state[1] must hold the gradient"
        t = float(r["before"]["ctr"][a, L.CTR_ALPHA] + 1)
        p1, m1, v1 = adam_ref(la0[a * 5], g, la0[a * 5 + 2], la0[a * 5 + 3], t, r["lr"][a])
        E_p, E_m, E_v = adam_bound(p1, m1, v1, g, la0[a * 5 + 2], t, r["lr"][a], 0.0, scalar=True)
        for i, (want, e, what) in enumerate(((p1, E_p, "log alpha"), (m1, E_m, "exp_avg"), (v1, E_v, "exp_avg_sq"))):
            got = r["la"][a, [0, 2, 3][i]].item()
            ratio = abs(got - want) / e
            WORST["fused alpha adam"] = max(WORST.get("fused alpha adam", 0.0), ratio)
            assert ratio <= 1.0, f"{tag} {what}: {got} vs {want} (bound {e})"
        alpha = math.exp(r["la"][a, 0].item())
        ratio = abs(r["out"][a, L.OUT_ALPHA].item() - alpha) / ((2 * EXP_ULP + 1) * U * alpha)
        WORST["fused alpha adam"] = max(WORST["fused alpha adam"], ratio)
        assert ratio <= 1.0, f"{tag}: out[ALPHA] {r['out'][a, L.OUT_ALPHA].item()} vs exp(log alpha) {alpha}"
        o_own[a, [L.OUT_ALPHA_LOSS, L.OUT_ALPHA]] = True
    _common_untouched(r, ws_own, r["tag"])
    untouched(r["eo_f"], what="eps2_out")
    untouched(r["o_f"], r["out"], ~o_own, "out")
    assert torch.isnan(r["la"][:, 4]).all() and torch.isnan(r["la_f"][:64]).all() and torch.isnan(r["la_f"][-64:]).all(), \
        "log alpha: alpha_kernel wrote past the four Adam fields"
    want = r["before"]["ctr"].clone()
    want[:, L.CTR_ALPHA] += 1
    assert torch.equal(r["ctr"], want), f"counters {r['ctr'].tolist()} != {want.tolist()} (ALPHA + 1, the ticket re-armed to 0)"
    assert torch.equal(_bits(r["rw_f"]), r["before"]["rw"]), "the rows changed"


ALPHA_CASES = [c for c in ACTOR_CASES if not SHAPES[c[0]][2] and "auto0" not in c[3]]


@pytest.mark.gpu
@pytest.mark.parametrize("shape,B,n,opts", ALPHA_CASES)
def test_alpha_kernel_matches_float64(shape, B, n, opts):
    """alpha_kernel alone (SAC): each tile's sum over its valid rows of -log pi - targ_ent (the agent's own targ_ent),
    alpha_loss, one Adam step of log alpha with the agent's lr, out[ALPHA], the counter and the re-armed ticket."""
    L = _lib()
    check_alpha(L, run_case(L, shape, B, n, opts, 4))


@pytest.mark.gpu
def test_fused_kernels_for_any_shape_and_option():
    """One derandomised draw over shapes, batches and options, each case through all three kernels."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as hs

    @hs.composite
    def cases(draw):
        shape = draw(hs.sampled_from(sorted(SHAPES)))
        B = draw(hs.sampled_from([1, 7, 9, 64, 255, 257, 1000, 2047]))
        n = draw(hs.sampled_from([1, 1, 2, 3]))
        opts = [x for x, on in (("ln0", draw(hs.booleans())), ("bcq", draw(hs.booleans())), ("smooth0", draw(hs.booleans())),
                                ("sym", draw(hs.booleans())), ("dev", draw(hs.booleans())), ("table", draw(hs.booleans()))) if on]
        return shape, B, n, ",".join(opts)

    @settings(max_examples=6, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(case=cases())
    def run(case):
        shape, B, n, opts = case
        L = _lib()
        check_critic(L, run_case(L, shape, B, n, opts, 0, seed=1))
        check_actor(L, run_case(L, shape, B, n, opts, 2, seed=1))
        if not SHAPES[shape][2]:
            check_alpha(L, run_case(L, shape, B, n, opts, 4, seed=1))

    run()


@pytest.mark.gpu
def test_report_worst_fused_ratios():
    """(runs after the tests above in this module) the worst deviation / bound ratio of each output kind, and the share of
    ReLU units (and arg-min rows) whose mask the interval treatment widened."""
    for k, v in sorted(WORST.items()):
        if k.startswith("fused"):
            print(f"worst dev/bound {k:28s} {v:.3f}")
    for k, (wide, tot, differ) in sorted(MASKS.items()):
        print(f"masks {k:40s} widened {wide} of {tot} ({wide / max(tot, 1):.2e}); kernel != float64 at {differ}")


# ---- the bounds have teeth (no GPU) ------------------------------------------------------------------------------------------
def _small_case(seed=0, td3=False, ln=True, B=20, O=3, A=2):
    """CPU inputs at a small shape: arena regions 0 / 1, a batch, noise, bounds."""
    from sac_td3_cudagraphs_pytorch_b200.arena import make_layout
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)
    lay = make_layout(O, A, td3, ln)
    P, T = torch.zeros(lay.region), torch.zeros(lay.region)
    for net in (*lay.critic, lay.actor):
        for f in ("w1t", "b1", "g1", "be1", "w2t", "b2", "g2", "be2", "w3", "b3"):
            if net.off[f] < 0:
                continue
            n_ = net.numel(f)
            scale = {"w1t": 1.5 / math.sqrt(net.in_dim), "w2t": 1 / 12.0, "w3": 1 / 12.0}.get(f, 0.2)
            v = rn(n_) * scale + (1.0 if f in ("g1", "g2") else 0.0)
            P[net.off[f]:net.off[f] + n_] = v
            T[net.off[f]:net.off[f] + n_] = v + 0.2 * scale * rn(n_)
    lo, hi = -0.5 - torch.rand(A, generator=g), 0.2 + torch.rand(A, generator=g)
    batch = (1.5 * rn(B, O), lo + (hi - lo) * torch.rand(B, A, generator=g), rn(B), (torch.rand(B, generator=g) < 0.3).float(),
             1.5 * rn(B, O))
    return lay, P, T, batch, rn(B, A), lo, hi


def _torch_net(X, p, dt):
    """One net in dtype dt with torch's own ops (another summation order): z1, z2 (leaves of autograd), h1, h2, out."""
    F = torch.nn.functional
    z1 = X.to(dt) @ p["w1t"].to(dt) + p["b1"].to(dt)
    if z1.requires_grad:
        z1.retain_grad()
    else:
        z1.requires_grad_()
    h1 = torch.relu(F.layer_norm(z1, (HID,), p["g1"].to(dt), p["be1"].to(dt), 1e-5) if p["ln"] else z1)
    z2 = h1 @ p["w2t"].to(dt) + p["b2"].to(dt)
    z2.retain_grad()
    h2 = torch.relu(F.layer_norm(z2, (HID,), p["g2"].to(dt), p["be2"].to(dt), 1e-5) if p["ln"] else z2)
    return z1, z2, h1, h2, h2 @ p["w3"].to(dt).T + p["b3"].to(dt)


def _torch_sample(u, eps, lo, hi, A, dt):
    """SAC's sample and log pi with torch ops; log N written as the kernel differentiates it (-eps^2 / 2 - log sigma)."""
    scale, bias = ((hi - lo) * 0.5).to(dt), ((hi + lo) * 0.5).to(dt)
    mu, raw = u[:, :A], u[:, A:2 * A]
    sigma = torch.exp(-5.0 + 3.5 * (torch.tanh(raw) + 1.0))
    y = torch.tanh(mu + eps.to(dt) * sigma)
    logp = (-0.5 * eps.to(dt) ** 2 - torch.log(sigma) - 0.9189385332046727 - torch.log(scale * (1 - y * y) + 1e-6)).sum(1)
    return y * scale + bias, logp


def test_fused_bounds_have_teeth():
    """At small shapes on the CPU: every bound accepts an fp32 evaluation with torch's ops and autograd, and rejects at least
    tenfold a' of the neighbouring row of the tile, Q' of one critic only, the target pass on online parameters and the
    online pass on target parameters, SAC's a' from the target actor and TD3's from the online one, another agent's gamma
    or td3_c, 2 / (8 nblk) for 2 / B, the LayerNorm backward without its mean terms or with another row's rstd, SAC's dQ/da
    of critic 1 left out, c_pi = alpha / (8 nblk), alpha_kernel counting padded rows or another agent's targ_ent, and a
    ReLU mask taken from the wrong layer."""
    B = 20  # three tiles, the last one ragged: 8 nblk = 24
    nb8 = RT * nblk_of(B)
    for td3 in (False, True):
        lay, P, T, batch, eps, lo, hi = _small_case(td3=td3, B=B)
        obs, act, rew, done, nobs = batch
        la, gamma, std, c = torch.tensor(-0.7, dtype=torch.float64), f32(0.97), f32(0.3), f32(0.4)
        tag = "td3" if td3 else "sac"
        # ---- critic step, fp32 with autograd: y, Q, h2, dz2, dz1 of critic 0 within the bounds of the kernel-masked reference
        pa32 = net_params(T if td3 else P, lay.actor)
        u = _torch_net(nobs, pa32, torch.float32)[4]
        if td3:
            a2 = torch.tanh(u) * ((hi - lo) * 0.5) + (hi + lo) * 0.5
            a2 = torch.minimum(torch.maximum(a2 + (eps * std).clamp(-c, c), lo), hi)
            lp2 = torch.zeros(B)
        else:
            a2, lp2 = _torch_sample(u, eps, lo, hi, lay.actor.out_dim // 2, torch.float32)
        qn = [_torch_net(torch.cat([nobs, a2], 1), net_params(T, lay.critic[k]), torch.float32)[4][:, 0] for k in range(2)]
        qp = torch.minimum(*qn) - (0.0 if td3 else math.exp(-0.7) * lp2)
        y32 = rew + (1.0 - done) * gamma * qp
        y32 = y32.detach()
        on = [_torch_net(torch.cat([obs, act], 1), net_params(P, lay.critic[k]), torch.float32) for k in range(2)]
        sum(((x[4][:, 0] - y32) ** 2).sum() for x in on).mul(1.0 / B).backward()
        kern = dict(y=y32, k=[dict(h1=x[2].detach(), h2=x[3].detach(), q=x[4][:, 0].detach(), dz3=(x[4][:, 0].detach() - y32) * (2.0 / B),
                                   dz2=x[1].grad, dz1=x[0].grad) for x in on])
        ref = critic_step_ref(P, T, lay, batch, eps, lo, hi, la, gamma, std, c, td3, False, True, kern)
        _fp32_within(f"{tag} y", y32, ref["y"])
        for k in range(2):
            rk, kk = ref["k"][k], kern["k"][k]
            _fp32_within(f"{tag} Q{k}", kk["q"], rk["q"])
            _fp32_within(f"{tag} dz3 {k}", kk["dz3"], rk["dz"])
            _fp32_within(f"{tag} h2 {k}", kk["h2"], rk["h2"])
            _fp32_within(f"{tag} dz2 {k}", kk["dz2"], rk["dz2"])
            _fp32_within(f"{tag} dz1 {k}", kk["dz1"], rk["dz1"])
        r0, k0 = ref["k"][0], kern["k"][0]
        # ---- critic step mistakes
        pol = next_action(net_params(T if td3 else P, lay.actor), nobs, eps, lo, hi, td3, True, std, c)
        qn_of = lambda act_, region: [q_pass(net_params(region, lay.critic[k]), rcat(nobs, act_))[1] for k in range(2)]
        y_of = lambda q0, q1, lp=pol.get("logp"), g_=gamma: q_target_ref(r0["q"], q0, q1, lp, la, rew, done, g_, B, td3, False)["y"].v
        nb = pol["act"].v[torch.arange(B) ^ 1]
        _teeth(f"{tag} y, a' of the neighbouring row", y_of(*qn_of(nb, T)), ref["y"])
        qt = qn_of(pol["act"], T)
        kw = int(bool((qt[1].v > qt[0].v).sum() > B // 2))  # (the critic whose Q' is the larger in most rows)
        _teeth(f"{tag} y, Q' of critic {kw} only", y_of(qt[kw], qt[kw]), ref["y"])
        _teeth(f"{tag} y, the target pass on online parameters", y_of(*qn_of(pol["act"], P)), ref["y"])
        _teeth(f"{tag} Q, the online pass on target parameters", q_pass(net_params(T, lay.critic[0]), torch.cat([obs, act], 1))[1].v,
               r0["q"])
        wrong_actor = next_action(net_params(P if td3 else T, lay.actor), nobs, eps, lo, hi, td3, True, std, c)
        _teeth(f"{tag} y, a' from the {'online' if td3 else 'target'} actor",
               y_of(*qn_of(wrong_actor["act"], T), lp=wrong_actor.get("logp")), ref["y"])
        _teeth(f"{tag} y, another agent's gamma", y_of(*qt, g_=f32(0.9)), ref["y"])
        if td3:
            other_c = next_action(net_params(T, lay.actor), nobs, eps * 4.0, lo, hi, td3, True, std, f32(0.05))
            this_c = next_action(net_params(T, lay.actor), nobs, eps * 4.0, lo, hi, td3, True, std, c)
            _teeth("td3 a', another agent's td3_c", other_c["act"].v, this_c["act"])
        _teeth(f"{tag} dz3, 2 / (8 nblk) for 2 / B", (k0["q"].double() - y32.double()) * (2.0 / nb8), r0["dz"])
        # the LayerNorm backward and the masks, on critic 0's backward pass
        po = net_params(P, lay.critic[0])
        layers = r0["layers"]
        m = [relu_mask(layers[i]["pre"], "teeth", k0["h" + str(i + 1)]) for i in range(2)]
        dh2 = R(k0["dz3"])[:, None] * po["w3"][0]
        dn = mask_mul(m[1], dh2).v
        l2 = layers[1]
        _teeth(f"{tag} dz2, LayerNorm backward without its mean terms", l2["rstd"].v[:, None] * dn * po["g2"].double(), r0["dz2"])
        dx = dn * po["g2"].double()
        full = (dx - dx.mean(1, keepdim=True)) - l2["xh"].v * (dx * l2["xh"].v).mean(1, keepdim=True)
        _teeth(f"{tag} dz2, another row's rstd", l2["rstd"].v.roll(1)[:, None] * full, r0["dz2"])
        _teeth(f"{tag} dz1, the mask of layer 2 used for layer 1", trunk_bwd(dh2, layers, po, [m[1], m[1]])[0].v, r0["dz1"])
        _teeth(f"{tag} dz2, the mask of layer 1 used for layer 2", trunk_bwd(dh2, layers, po, [m[0], m[0]])[1].v, r0["dz2"])
        # ---- actor step, fp32 with autograd: the head gradient and the actor's dz1
        pa = net_params(P, lay.actor)
        z1, z2, h1, h2, u = _torch_net(obs, pa, torch.float32)
        z2.retain_grad()
        u.retain_grad()
        A = lo.shape[0]
        if td3:
            api = torch.tanh(u) * ((hi - lo) * 0.5) + (hi + lo) * 0.5
            loss = -_torch_net(torch.cat([obs, api], 1), net_params(P, lay.critic[0]), torch.float32)[4][:, 0]
        else:
            api, lpi = _torch_sample(u, eps, lo, hi, A, torch.float32)
            qq = [_torch_net(torch.cat([obs, api], 1), net_params(P, lay.critic[k]), torch.float32)[4][:, 0] for k in range(2)]
            loss = math.exp(-0.7) * lpi - torch.minimum(*qq)
        loss.mean().backward()
        kern = dict(h1=h1.detach(), h2=h2.detach(), dz3=u.grad, dz2=z2.grad, dz1=z1.grad)
        ra = actor_step_ref(P, lay, obs, eps, lo, hi, la, td3, kern)
        _fp32_within(f"{tag} actor h2", h2.detach(), ra["h2"])
        _fp32_within(f"{tag} actor dz3", u.grad, ra["du"])
        _fp32_within(f"{tag} actor dz2", z2.grad, ra["dz2"])
        _fp32_within(f"{tag} actor dz1", z1.grad, ra["dz1"])
        _fp32_within(f"{tag} actor loss partials", group_sum(R(loss.detach().double()[:, None]), RT, 0).v[:, 0], ra["loss"])
        if not td3:
            sv = [ra["pol"][f] for f in ("eps", "sigma", "y", "th")]
            wrong = head_bwd_ref(ra["da"][0], None, sv, lo, hi, la, False, A, B, recip=True)
            _teeth("sac actor dz3, dQ/da of critic 1 left out", wrong["du"].v, ra["du"])
            wrong = actor_step_ref(P, lay, obs, eps, lo, hi, la, td3, kern, c_pi_rows=nb8)
            _teeth("sac actor dz3, c_pi = alpha / (8 nblk)", wrong["du"].v, ra["du"])
            # ---- alpha_kernel
            t32 = -lpi.detach() - f32(-2.0)
            ref_a = alpha_terms_ref(P, lay, obs, eps, lo, hi, -2.0)
            _fp32_within("alpha partials", group_sum(R(t32.double()[:, None]), RT, 0).v[:, 0], ref_a["part"])
            padded = torch.cat([ref_a["t"].v, torch.full((nb8 - B,), -f32(-2.0), dtype=torch.float64)])  # (-0 - targ_ent)
            _teeth("alpha partials, padded rows counted", padded.view(-1, RT).sum(1), ref_a["part"])
            _teeth("alpha partials, another agent's targ_ent", alpha_terms_ref(P, lay, obs, eps, lo, hi, -3.0)["part"].v, ref_a["part"])
