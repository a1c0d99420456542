"""The wide (layer-by-layer, tensor-core) update for LARGE batches (BASELINE.json config 5) and for STACKED agents
(config 4).

``Agent.update_qnets`` / ``update_actor`` (agents/agent.py:183-318) restated as a sequence of batch-parallel kernels
(csrc/wide.cu) around the tcgen05 hidden layers (csrc/tc_linear.cu, csrc/tc_wgrad.cu): the row-group kernels that win
at batch 256 stream every layer's weights from L2 once per 8 rows and stay at ~10 TFLOP/s however large the batch is;
here weights are read once per 128 rows (TMA) and the 256x256 products — forward, dX and weight gradients — run on the
tensor cores. Precision "3xtf32" (default) splits every operand into a TF32 hi and lo part and issues three MMAs per
product: fp32-level accuracy (gradients within 2e-5 of the oracle, tests/test_gpu_wide.py); "tf32" is the plain,
~1e-3-per-product mode (the north star's "looser stated bound"). Everything outside the products (LayerNorm, heads, TD
target, losses, optimizer) is fp32 and the Philox noise is keyed exactly as in the row path, so both paths draw the same
samples. The owner is an ``Agent`` (one learner) or a ``population.Population`` (n learners stacked along the rows of the
same launches: include/b2rl.h, b2rl_stack_t).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L

STREAM_CRITIC_EPS, STREAM_ACTOR_EPS, STREAM_ALPHA_EPS = 1, 2, 3  # csrc/rng.cuh


class _Owner:
    """What the wide path needs from its owner, which is either an ``Agent`` (one learner: every array has M rows, the
    C ABI's ``stack`` argument is NULL) or a ``population.Population`` (N stacked learners, BASELINE.json config 4: every
    per-row array is [N][M][..], parameters / scalars are reached through the strides of ``b2rl_stack_t``)."""

    def __init__(self, owner):
        self.owner = owner
        self.stacked = hasattr(owner, "N")  # a Population
        self.lib, self.device, self.layout, self.arena = owner._lib, owner.device, owner.layout, owner.arena
        self.fmt, self.hps, self.hyper, self.td3, self.ac_dim = owner.fmt, owner.hps, owner._hyper, owner.td3, owner.ac_dim
        self.min_ac, self.max_ac, self.counters, self.out = owner.min_ac, owner.max_ac, owner.counters, owner.out
        self.autotune = owner.autotune
        if self.stacked:
            self.n, self.base, self.alpha_state = owner.N, owner.base, owner.alpha_state
            self.launch_adam = owner._adam
        else:
            self.n, self.base, self.alpha_state = 1, owner.agent_id, owner._alpha_state
            self.launch_adam = owner._launch_adam
        self._stk = None
        self._ws = {}

    def stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def stack(self, lo_stride: int = 0):
        """The ``b2rl_stack_t*`` argument (None for a single learner)."""
        if not self.stacked:
            return None
        return L.Stack(self.n, self.base, self.arena.agent_stride, lo_stride, self.alpha_state.stride(0), self.counters.stride(0),
                       self.out.stride(0), self.owner.agent_hp_table.data_ptr())

    def workspace(self, M: int) -> torch.Tensor:
        """H1 H2 DZ1 DZ2 [2][n*M][256] + DZ3 [2][n*M][MAX_OUT], shared by the critic and the actor step."""
        if not self.stacked:
            return self.owner.workspace(M)
        if M not in self._ws:
            nm = self.n * M
            self._ws[M] = torch.zeros(8 * nm * 256 + 2 * nm * L.MAX_OUT, dtype=torch.float32, device=self.device)
        return self._ws[M]

    def lo_mirror(self) -> torch.Tensor:
        """[n][2][region] lo parts of the online / target regions (3xTF32), maintained by the owner's Adam launches."""
        return self.owner.lo_mirror()

    def seg(self, begin, end, lr, adam, polyak, counter=0, clip=False):
        return L.Seg(begin, end, lr, int(adam), int(polyak), counter, 1.0, int(clip))


def _first_layer(lib, x_ptr, ldx, M, K, w1t, b, g, be, ln, H, XH, stat, x3, stk, st):
    """First layer of a network (agents/nets.py:66-72): on the tensor cores (tc_linear.cu MODE 1) when TMA can address the
    rows' inputs (16-byte aligned, pitch a multiple of 4 floats), else the FFMA kernel of wide.cu."""
    import os
    if x_ptr % 16 == 0 and ldx % 4 == 0 and os.environ.get("B2RL_WIDE_FIRST", "tc") == "tc":
        L.check(lib.b2rl_tc_first(x_ptr, ldx, M, K, w1t, b, g, be, ln, H, XH, stat, x3, stk, st), "tc_first")
    else:
        L.check(lib.b2rl_wide_first(x_ptr, ldx, M, K, w1t, b, g, be, ln, H, XH, stat, stk, st), "wide_first")


def _tc_wgrads(lib, stk, M, x3, scratch, G, net, x0_ptr, ldx, h1, h2, dz1, dz2, dz3, bump, st, w3_done=False):
    """dW1t = X0^T dZ1, dW2t = H1^T dZ2, dW3 = dZ3^T H2 of one network, on the tensor cores (tc_wgrad.cu) into the arena's
    gradient region at G. w3_done: the scalar head's gradient came out of wide_ln_bwd already (critics)."""
    o = net.off
    f = lambda off: G + 4 * off
    sc = scratch.data_ptr()
    L.check(lib.b2rl_tc_wgrad(x0_ptr, ldx, ldx, net.in_dim, dz1, M, f(o["w1t"]), None, sc, x3, None, stk, st), "tc_wgrad w1")
    # (no transposed copy into the w2n shadow's gradient: the Adam launch derives the shadow from w2t, adam.cu)
    L.check(lib.b2rl_tc_wgrad(h1, 256, 256, 256, dz2, M, f(o["w2t"]), None, sc, x3, bump if w3_done else None, stk, st), "tc_wgrad w2")
    if not w3_done:
        L.check(lib.b2rl_tc_wgrad(dz3, L.MAX_OUT, L.MAX_OUT, net.out_dim, h2, M, f(o["w3"]), None, sc, x3, bump, stk, st), "tc_wgrad w3")


def _colsums(lib, jobs, P, G, stk, st):
    """All column-sum reductions of a step in one launch (b2rl_wide_colsum_multi): jobs = [(part_ptr, off_b, off_g, off_be, ln)].
    Their producers differ (wide_ln_bwd, tc_linear_bwd), their only consumer is the optimizer launch."""
    arr = (L.ColsumJob * len(jobs))()
    for a, (part, ob, og, obe, ln) in zip(arr, jobs):
        a.part, a.off_b, a.off_g, a.off_be, a.layer_norm = part, ob, og, obe, int(ln)
    L.check(lib.b2rl_wide_colsum_multi(arr, len(jobs), P, G, stk, st), "wide_colsum_multi")


def _wgrad_scratch(own: "_Owner", M):
    dims = {1, 256} | {n.in_dim for n in [own.layout.actor, *own.layout.critic]}
    n = own.n if own.stacked else 0
    return torch.empty(max(own.lib.b2rl_tc_wgrad_scratch_floats(d, M, n) for d in dims), dtype=torch.float32, device=own.device)


class WideCritic:
    def __init__(self, agent, batch: int, precision: str = "3xtf32"):
        """precision: "3xtf32" (default; hi/lo operand split, three MMAs per product: fp32-level accuracy) or "tf32"
        (single MMA, ~1e-3 per product, ~1e-2 on gradients because dLoss/dQ is a difference of Q and the TD target)."""
        assert precision in ("3xtf32", "tf32")
        self.x3 = precision == "3xtf32"
        own = self.ag = agent if isinstance(agent, _Owner) else _Owner(agent)  # an Agent, or a Population (M rows PER AGENT)
        self.M = int(batch)
        M, dev, n = self.M, own.device, own.n
        NM = self.NM = n * M  # rows of the stacked arrays
        self._lib = own.lib
        f32 = dict(dtype=torch.float32, device=dev)
        O, A = own.fmt.ob_dim, own.ac_dim
        self.ldn = (O + A + 3) & ~3
        self.t1, self.t2 = torch.empty(NM, 256, **f32), torch.empty(NM, 256, **f32)     # scratch activations
        self.xn = torch.zeros(NM, self.ldn, **f32)                                       # [next_obs | a']
        self.logp, self.qn, self.q = torch.zeros(NM, **f32), torch.zeros(2, NM, **f32), torch.zeros(2, NM, **f32)
        self.xh1, self.xh2 = torch.empty(2, NM, 256, **f32), torch.empty(2, NM, 256, **f32)
        self.st1, self.st2 = torch.zeros(2, NM, 2, **f32), torch.zeros(2, NM, 2, **f32)
        self.P128, self.P8 = (M + 127) // 128, (M + 7) // 8   # per agent
        self.part1, self.part2 = torch.zeros(2, n * self.P128, 3, 256, **f32), torch.zeros(2, n * self.P128, 3, 256, **f32)
        self.part3 = torch.zeros(2, n * self.P128, 3, 256, **f32)  # slot 0: per-CTA partials of the critics' head gradient
        self.sq = torch.zeros(2, n * self.P8, 2, **f32)  # per-CTA {sum sq err, sum dQ} of wide_q_head
        self.ws = own.workspace(M)
        # lo parts (3xTF32) of the weights. One learner: a [2][region] mirror of the online and target regions at the
        # parameters' own offsets, created (and filled) here, kept current from now on by the owner's Adam / Polyak launches —
        # no split pass per step. Stacked agents: no mirror at all — every weight slab serves one tile pair, so the kernel
        # splits it in shared memory (W_lo == W, include/b2rl.h) and 268 MB of reads per launch and the optimizer's mirror
        # writes (2.2 of 9.4 MB per agent and critic step) disappear.
        self.wlo = own.lo_mirror() if (self.x3 and not own.stacked) else None
        self.stk = own.stack(lo_stride=2 * own.layout.region)
        self.gscratch = _wgrad_scratch(own, M)

    # pointers into the arena (agent 0's copy): region r, float offset o
    def _p(self, region: int, off: int) -> int:
        return self.ag.arena.flat.data_ptr() + 4 * (region * self.ag.layout.region + off)

    def _ws(self, which: int, slot: int) -> int:  # H1 H2 DZ1 DZ2 of common.cuh::ws_carve
        return self.ws.data_ptr() + 4 * ((which * 2 + slot) * self.NM * 256)

    def _dz3(self, slot: int) -> int:
        return self.ws.data_ptr() + 4 * (8 * self.NM * 256 + slot * self.NM * L.MAX_OUT)

    def update_qnets(self, rows: torch.Tensor, eps: Optional[torch.Tensor] = None, eps_out: Optional[torch.Tensor] = None,
                     targ_out: Optional[torch.Tensor] = None, adam: bool = True, polyak: bool = False, extra_segs=()) -> dict:
        """rows: the sampled batch [M][row_stride] (replay.Batch.rows; stacked: [n_agents][M][row_stride]).
        Enqueue-only (graph-capturable). adam=False: stop after the gradients (data parallel: all-reduce them, then step);
        polyak / extra_segs: let the target average ride in the Adam launch (population.py)."""
        ag, lib, M = self.ag, self._lib, self.M
        assert rows.numel() == self.NM * ag.fmt.row_stride and rows.is_contiguous()
        lay, st = ag.layout, ag.stream()
        O, A, rs = ag.fmt.ob_dim, ag.ac_dim, ag.fmt.row_stride
        ln = int(bool(ag.hps.layer_norm))
        RP, RT, RG = L.REGION_P, L.REGION_T, 4
        none = None
        stk = C.byref(self.stk) if self.stk is not None else None

        def first(x_ptr, ldx, K, net, region, H, XH, stat):
            o = net.off
            _first_layer(lib, x_ptr, ldx, M, K, self._p(region, o["w1t"]), self._p(region, o["b1"]),
                         self._p(region, o["g1"]) if ln else none, self._p(region, o["be1"]) if ln else none, ln,
                         H, XH, stat, int(self.x3), stk, st)

        # every weight keeps its arena offset in the lo mirror (3xTF32), which the optimizer launches keep current
        base = self._p(RP, 0)
        ra = RT if ag.td3 else RP  # next action: SAC samples from the ONLINE actor (agent.py:205), TD3 uses the TARGET actor
        act = lay.actor

        def lo_of(slot, w_ptr):
            if not self.x3:
                return none
            return w_ptr if self.wlo is None else self.wlo.data_ptr() + (w_ptr - base)

        def hidden(x_ptr, net, region, H, XH, stat, slot, head=None):
            o = net.off
            w = self._p(region, o["w2n"])
            b2, g2, be2 = self._p(region, o["b2"]), self._p(region, o["g2"]) if ln else none, self._p(region, o["be2"]) if ln else none
            if head is None:
                L.check(lib.b2rl_tc_linear(x_ptr, 256, M, w, lo_of(slot, w), b2, g2, be2, ln, 1, H, XH, stat, stk, st), "tc_linear")
            else:  # the critic's scalar head in the same kernel's epilogue
                L.check(lib.b2rl_tc_linear_q(x_ptr, 256, M, w, lo_of(slot, w), b2, g2, be2, ln, H, XH, stat, C.byref(head), stk, st),
                        "tc_linear_q")

        # ---- next action (agent.py:194-205)
        first(rows.data_ptr() + 4 * (O + A + 2), rs, O, act, ra, self.t1.data_ptr(), none, none)
        hidden(self.t1.data_ptr(), act, ra, self.t2.data_ptr(), none, none, 0)
        p = L.WidePolicy()
        p.h2, p.w3, p.b3 = self.t2.data_ptr(), self._p(ra, act.off["w3"]), self._p(ra, act.off["b3"])
        p.rows, p.min_ac, p.max_ac = rows.data_ptr(), ag.min_ac.data_ptr(), ag.max_ac.data_ptr()
        p.eps, p.eps_out, p.xn = L.ptr(eps), L.ptr(eps_out), self.xn.data_ptr()
        p.logp = None if ag.td3 else self.logp.data_ptr()
        p.counters = ag.counters.data_ptr()
        p.M, p.O, p.A, p.out_dim, p.row_stride, p.ldn, p.src_off = M, O, A, act.out_dim, rs, self.ldn, O + A + 2
        p.td3, p.smoothing = int(ag.td3), int(ag.hyper.targ_smoothing)
        p.counter_idx, p.stream_id = L.CTR_Q, STREAM_CRITIC_EPS
        p.td3_std, p.td3_c, p.seed, p.agent = ag.hyper.td3_std, ag.hyper.td3_c, ag.hyper.seed, ag.base
        L.check(lib.b2rl_wide_policy_head(C.byref(p), stk, st), "wide_policy_head")

        def q_head(net, region, k, mode):
            q = L.WideQ()
            q.h2, q.w3, q.b3 = None, self._p(region, net.off["w3"]), self._p(region, net.off["b3"])
            q.q_out = (self.q if mode else self.qn)[k].data_ptr()
            q.qn0, q.qn1, q.logp = self.qn[0].data_ptr(), self.qn[1].data_ptr(), self.logp.data_ptr()
            q.rows, q.log_alpha = rows.data_ptr(), ag.alpha_state.data_ptr()
            q.dz3, q.sq_part = self._dz3(k), self.sq[k].data_ptr()
            q.targ_out = L.ptr(targ_out) if (mode and k == 0) else None
            q.M, q.mode, q.row_stride, q.rd_off, q.td3, q.bcq_mix = M, mode, rs, O + A, int(ag.td3), int(ag.hyper.bcq_mix)
            q.gamma = ag.hyper.gamma
            return q

        # ---- twin target Q on (next_obs, a')  (agent.py:208-210)
        for k in range(2):
            net = lay.critic[k]
            first(self.xn.data_ptr(), self.ldn, O + A, net, RT, self.t1.data_ptr(), none, none)
            hidden(self.t1.data_ptr(), net, RT, none, none, none, 1 + k, head=q_head(net, RT, k, 0))  # (h2 stays on chip)
        # ---- twin online Q, TD target, loss, backward (agent.py:212-235)
        G = self._p(RG, 0)
        jobs = []
        for k in range(2):
            net, o = lay.critic[k], lay.critic[k].off
            first(rows.data_ptr(), rs, O + A, net, RP, self._ws(0, k), self.xh1[k].data_ptr(), self.st1[k].data_ptr())
            # (h2 itself never goes to memory: the head rides in the epilogue and its weight gradient is rebuilt from x-hat
            # inside wide_ln_bwd; only x-hat and the statistics are kept for the backward pass)
            hidden(self._ws(0, k), net, RP, none, self.xh2[k].data_ptr(), self.st2[k].data_ptr(), 3 + k,
                   head=q_head(net, RP, k, 1))
            L.check(lib.b2rl_wide_ln_bwd(self._dz3(k), 1, self._p(RP, o["w3"]), self.xh2[k].data_ptr(), self.st2[k].data_ptr(),
                                         self._p(RP, o["g2"]) if ln else none, self._p(RP, o["be2"]) if ln else none, ln, M,
                                         self._ws(3, k), self.part2[k].data_ptr(), self.part3[k].data_ptr(), stk, st), "wide_ln_bwd")
            jobs.append((self.part3[k].data_ptr(), o["w3"], 0, 0, 0))  # dW3
            w2t = self._p(RP, o["w2t"])
            L.check(lib.b2rl_tc_linear_bwd(self._ws(3, k), M, w2t, lo_of(5 + k, w2t), self.xh1[k].data_ptr(), self.st1[k].data_ptr(),
                                           self._p(RP, o["g1"]) if ln else none, self._p(RP, o["be1"]) if ln else none, ln,
                                           self._ws(2, k), self.part1[k].data_ptr(), stk, st), "tc_linear_bwd")
            jobs.append((self.part2[k].data_ptr(), o["b2"], o["g2"] if ln else 0, o["be2"] if ln else 0, ln))
            jobs.append((self.part1[k].data_ptr(), o["b1"], o["g1"] if ln else 0, o["be1"] if ln else 0, ln))
        _colsums(lib, jobs, self.P128, G, stk, st)
        L.check(lib.b2rl_wide_critic_scalars(self.sq[0].data_ptr(), self.sq[1].data_ptr(), self.P8, self._dz3(0), self._dz3(1), M, G,
                                             lay.critic[0].off["b3"], lay.critic[1].off["b3"], ag.out.data_ptr(), stk, st),
                "wide_critic_scalars")
        # ---- weight gradients (wgrad.cu reads rows / H1 / H2 / DZ1 / DZ2 / DZ3 of the workspace), then Adam
        for k in range(2):
            _tc_wgrads(lib, stk, M, int(self.x3), self.gscratch, G, lay.critic[k], rows.data_ptr(), rs, self._ws(0, k), self._ws(1, k),
                       self._ws(2, k), self._ws(3, k), self._dz3(k), ag.counters.data_ptr() + 8 * L.CTR_Q if k == 1 else None, st,
                       w3_done=True)
        if adam:
            ag.launch_adam([ag.seg(lay.critic[0].begin, lay.critic[1].end, float(ag.hps.qnets_lr), True, polyak, L.CTR_Q)]
                           + list(extra_segs))
        return {"loss/qf_loss": ag.out[..., L.OUT_QF_LOSS]}


class WideActor:
    """``Agent.update_actor`` (agents/agent.py:244-318) on the wide path: actor forward, sample, twin Q with the
    critics' parameters held constant, loss, backward through the arg-min critic down to its action inputs
    (dQ/da), through the action head and the actor's two layers, weight gradients, Adam; then SAC's temperature
    step with the UPDATED actor and fresh noise. Same conventions as WideCritic. Gradient clipping
    (hps.clip_norm > 0) is not offered on this path."""

    def __init__(self, agent, batch: int, precision: str = "3xtf32"):
        assert precision in ("3xtf32", "tf32")
        own = self.ag = agent if isinstance(agent, _Owner) else _Owner(agent)
        assert not (own.owner._clip if own.stacked else own.hps.clip_norm > 0), \
            "the wide actor step has no gradient clipping: use the row-group path"
        self.x3 = precision == "3xtf32"
        self.M = int(batch)
        M, dev, n = self.M, own.device, own.n
        NM = self.NM = n * M
        self._lib = own.lib
        f32 = dict(dtype=torch.float32, device=dev)
        O, A = own.fmt.ob_dim, own.ac_dim
        self.ldn = (O + A + 3) & ~3
        self.nq = 1 if own.td3 else 2  # TD3's loss uses critic 0 only (agent.py:274-275)
        self.t1, self.t2 = torch.empty(NM, 256, **f32), torch.empty(NM, 256, **f32)
        self.xq = torch.zeros(NM, self.ldn, **f32)                       # [obs | a_pi]
        self.save = torch.zeros(NM, 4, A, **f32)
        self.logp, self.logp2 = torch.zeros(NM, **f32), torch.zeros(NM, **f32)
        self.q = torch.zeros(2, NM, **f32)
        self.xa1, self.xa2 = torch.empty(NM, 256, **f32), torch.empty(NM, 256, **f32)       # actor x-hat
        self.sa1, self.sa2 = torch.zeros(NM, 2, **f32), torch.zeros(NM, 2, **f32)
        self.xq1, self.xq2 = torch.empty(2, NM, 256, **f32), torch.empty(2, NM, 256, **f32)  # critics' x-hat
        self.sq1, self.sq2 = torch.zeros(2, NM, 2, **f32), torch.zeros(2, NM, 2, **f32)
        self.dzq = torch.zeros(2, NM, L.MAX_OUT, **f32)
        self.dqda = torch.zeros(2, NM, A, **f32)
        self.P128, self.P256 = (M + 127) // 128, (M + 255) // 256  # per agent
        self.part = torch.zeros(2, n * self.P128, 3, 256, **f32)
        self.part_s, self.part_du = torch.zeros(n * self.P256, 2, **f32), torch.zeros(n * self.P256, L.MAX_OUT, **f32)
        self.ws = own.workspace(M)
        self.wlo = own.lo_mirror() if (self.x3 and not own.stacked) else None  # (shared with WideCritic; see there)
        self.stk = own.stack(lo_stride=2 * own.layout.region)
        self.gscratch = _wgrad_scratch(own, M)

    _p = WideCritic._p
    _ws = WideCritic._ws
    _dz3 = WideCritic._dz3

    def update_actor(self, rows: torch.Tensor, eps: Optional[torch.Tensor] = None, eps_alpha: Optional[torch.Tensor] = None,
                     adam: bool = True, polyak: bool = False) -> dict:
        ag, lib, M = self.ag, self._lib, self.M
        assert rows.numel() == self.NM * ag.fmt.row_stride and rows.is_contiguous()
        lay, st = ag.layout, ag.stream()
        O, A, rs = ag.fmt.ob_dim, ag.ac_dim, ag.fmt.row_stride
        ln = int(bool(ag.hps.layer_norm))
        RP, RG = L.REGION_P, 4
        none = None
        act, ao = lay.actor, lay.actor.off
        la = ag.alpha_state.data_ptr()
        stk = C.byref(self.stk) if self.stk is not None else None

        def first(x_ptr, ldx, K, net, H, XH, stat):
            o = net.off
            _first_layer(lib, x_ptr, ldx, M, K, self._p(RP, o["w1t"]), self._p(RP, o["b1"]),
                         self._p(RP, o["g1"]) if ln else none, self._p(RP, o["be1"]) if ln else none, ln,
                         H, XH, stat, int(self.x3), stk, st)

        base = self._p(RP, 0)

        def lo_of(slot, w_ptr):
            if not self.x3:
                return none
            return w_ptr if self.wlo is None else self.wlo.data_ptr() + (w_ptr - base)

        def hidden(x_ptr, net, H, XH, stat, slot):
            o = net.off
            w = self._p(RP, o["w2n"])
            L.check(lib.b2rl_tc_linear(x_ptr, 256, M, w, lo_of(slot, w), self._p(RP, o["b2"]),
                                       self._p(RP, o["g2"]) if ln else none, self._p(RP, o["be2"]) if ln else none, ln, 1,
                                       H, XH, stat, stk, st), "tc_linear")

        def policy(h2_ptr, eps_t, stream_id, xn, logp, save):
            p = L.WidePolicy()
            p.h2, p.w3, p.b3 = h2_ptr, self._p(RP, ao["w3"]), self._p(RP, ao["b3"])
            p.rows, p.min_ac, p.max_ac = rows.data_ptr(), ag.min_ac.data_ptr(), ag.max_ac.data_ptr()
            p.eps, p.eps_out, p.xn, p.logp, p.save = L.ptr(eps_t), None, xn, logp, save
            p.counters = ag.counters.data_ptr()
            p.M, p.O, p.A, p.out_dim, p.row_stride, p.ldn, p.src_off = M, O, A, act.out_dim, rs, self.ldn, 0
            p.td3, p.smoothing, p.counter_idx, p.stream_id = int(ag.td3), 0, L.CTR_PI, stream_id
            p.td3_std, p.td3_c, p.seed, p.agent = 0.0, 0.0, ag.hyper.seed, ag.base
            L.check(lib.b2rl_wide_policy_head(C.byref(p), stk, st), "wide_policy_head")

        def bwd_layers(dz3_ptr, n_out, net, xh2, st2, xh1, st1, dz2_out, dz1_out, part, slot):
            o = net.off
            L.check(lib.b2rl_wide_ln_bwd(dz3_ptr, n_out, self._p(RP, o["w3"]), xh2, st2,
                                         self._p(RP, o["g2"]) if ln else none, self._p(RP, o["be2"]) if ln else none, ln, M,
                                         dz2_out, part[0].data_ptr() if part is not None else None, None, stk, st), "wide_ln_bwd")
            w2t = self._p(RP, o["w2t"])
            L.check(lib.b2rl_tc_linear_bwd(dz2_out, M, w2t, lo_of(slot, w2t), xh1, st1,
                                           self._p(RP, o["g1"]) if ln else none, self._p(RP, o["be1"]) if ln else none, ln,
                                           dz1_out, part[1].data_ptr() if part is not None else None, stk, st), "tc_linear_bwd")

        # ---- actor forward on obs, sample (agent.py:251 / :254-255): H1 / H2 go to workspace slot 0 for wgrad
        first(rows.data_ptr(), rs, O, act, self._ws(0, 0), self.xa1.data_ptr(), self.sa1.data_ptr())
        hidden(self._ws(0, 0), act, self._ws(1, 0), self.xa2.data_ptr(), self.sa2.data_ptr(), 0)
        policy(self._ws(1, 0), eps, STREAM_ACTOR_EPS, self.xq.data_ptr(), None if ag.td3 else self.logp.data_ptr(),
               self.save.data_ptr())
        # ---- Q_k(obs, a_pi) with the critics' parameters held constant (agent.py:272-278)
        for k in range(self.nq):
            net = lay.critic[k]
            first(self.xq.data_ptr(), self.ldn, O + A, net, self.t1.data_ptr(), self.xq1[k].data_ptr(), self.sq1[k].data_ptr())
            q = L.WideQ()  # the scalar head rides in the hidden layer's epilogue; h2 itself is not needed (x-hat is, for the backward)
            q.h2, q.w3, q.b3 = None, self._p(RP, net.off["w3"]), self._p(RP, net.off["b3"])
            q.q_out, q.M, q.mode = self.q[k].data_ptr(), M, 0
            o = net.off
            w2 = self._p(RP, o["w2n"])
            L.check(lib.b2rl_tc_linear_q(self.t1.data_ptr(), 256, M, w2, lo_of(1 + k, w2), self._p(RP, o["b2"]),
                                         self._p(RP, o["g2"]) if ln else none, self._p(RP, o["be2"]) if ln else none, ln, None,
                                         self.xq2[k].data_ptr(), self.sq2[k].data_ptr(), C.byref(q), stk, st), "tc_linear_q")
        L.check(lib.b2rl_wide_actor_loss(self.q[0].data_ptr(), None if ag.td3 else self.q[1].data_ptr(),
                                         None if ag.td3 else self.logp.data_ptr(), None if ag.td3 else la, int(ag.td3), M,
                                         self.dzq[0].data_ptr(), None if ag.td3 else self.dzq[1].data_ptr(),
                                         self.part_s.data_ptr(), stk, st), "wide_actor_loss")
        # ---- backward through critic k down to its action inputs
        for k in range(self.nq):
            net = lay.critic[k]
            bwd_layers(self.dzq[k].data_ptr(), 1, net, self.xq2[k].data_ptr(), self.sq2[k].data_ptr(), self.xq1[k].data_ptr(),
                       self.sq1[k].data_ptr(), self.t1.data_ptr(), self.t2.data_ptr(), None, 3 + k)  # (dX only: no column sums)
            L.check(lib.b2rl_wide_dqda(self.t2.data_ptr(), self._p(RP, net.off["w1t"]) + 4 * O * 256, A, M,
                                       self.dqda[k].data_ptr(), stk, st), "wide_dqda")
        # ---- backward through the action head and the actor
        G = self._p(RG, 0)
        L.check(lib.b2rl_wide_actor_head_bwd(self.dqda[0].data_ptr(), None if ag.td3 else self.dqda[1].data_ptr(),
                                             self.save.data_ptr(), ag.min_ac.data_ptr(), ag.max_ac.data_ptr(),
                                             None if ag.td3 else la, int(ag.td3), A, M, self._dz3(0), self.part_du.data_ptr(), stk, st),
                "wide_actor_head_bwd")
        bwd_layers(self._dz3(0), act.out_dim, act, self.xa2.data_ptr(), self.sa2.data_ptr(), self.xa1.data_ptr(),
                   self.sa1.data_ptr(), self._ws(3, 0), self._ws(2, 0), self.part, 5)
        _colsums(lib, [(self.part[0].data_ptr(), ao["b2"], ao["g2"] if ln else 0, ao["be2"] if ln else 0, ln),
                       (self.part[1].data_ptr(), ao["b1"], ao["g1"] if ln else 0, ao["be1"] if ln else 0, ln)], self.P128, G, stk, st)
        L.check(lib.b2rl_wide_actor_scalars(self.part_s.data_ptr(), self.part_du.data_ptr(), self.P256, M, act.out_dim,
                                            int(ag.td3), None if ag.td3 else la, G, ao["b3"], ag.out.data_ptr(), stk, st),
                "wide_actor_scalars")
        _tc_wgrads(lib, stk, M, int(self.x3), self.gscratch, G, act, rows.data_ptr(), rs, self._ws(0, 0), self._ws(1, 0),
                   self._ws(2, 0), self._ws(3, 0), self._dz3(0), ag.counters.data_ptr() + 8 * L.CTR_PI, st)
        if not adam:
            return {}
        ag.launch_adam([ag.seg(act.begin, act.end, float(ag.hps.actor_lr), True, polyak, L.CTR_PI)])
        out = {"loss/actor_loss": ag.out[..., L.OUT_ACTOR_LOSS]}
        if ag.td3:
            return out
        if ag.autotune:
            self.alpha_grad(rows, eps_alpha)
            if ag.stacked:  # the population's per-agent rates
                L.check(lib.b2rl_alpha_adam_hp(la, ag.counters.data_ptr(), ag.n, ag.owner.agent_hp_table.data_ptr(), 1.0,
                                               ag.out.data_ptr(), st), "alpha_adam_hp")
            else:
                L.check(lib.b2rl_alpha_adam(la, ag.counters.data_ptr(), ag.n, float(ag.hps.log_alpha_lr), 1.0, ag.out.data_ptr(), st),
                        "alpha_adam")
            out["loss/alpha_loss"] = ag.out[..., L.OUT_ALPHA_LOSS]
        out["vitals/alpha"] = ag.out[..., L.OUT_ALPHA]
        return out

    def alpha_grad(self, rows: torch.Tensor, eps_alpha: Optional[torch.Tensor] = None) -> None:
        """agents/agent.py:295-300: log-prob of a fresh sample from the UPDATED actor; leaves the temperature's
        gradient in its state slot 1 (finish with b2rl_alpha_adam, after an all-reduce when data parallel)."""
        ag, lib, M = self.ag, self._lib, self.M
        st, lay = ag.stream(), ag.layout
        O, rs = ag.fmt.ob_dim, ag.fmt.row_stride
        ln = int(bool(ag.hps.layer_norm))
        act, o, RP = lay.actor, lay.actor.off, L.REGION_P
        none = None
        stk = C.byref(self.stk) if self.stk is not None else None
        _first_layer(lib, rows.data_ptr(), rs, M, O, self._p(RP, o["w1t"]), self._p(RP, o["b1"]),
                     self._p(RP, o["g1"]) if ln else none, self._p(RP, o["be1"]) if ln else none, ln,
                     self.t1.data_ptr(), none, none, int(self.x3), stk, st)
        w = self._p(RP, o["w2n"])
        wl = none  # 3xTF32: the mirror the actor's Adam launch has just refreshed, or (stacked) the in-kernel split
        if self.x3:
            wl = w if self.wlo is None else self.wlo.data_ptr() + (w - self._p(RP, 0))
        L.check(lib.b2rl_tc_linear(self.t1.data_ptr(), 256, M, w, wl, self._p(RP, o["b2"]), self._p(RP, o["g2"]) if ln else none,
                                   self._p(RP, o["be2"]) if ln else none, ln, 1, self.t2.data_ptr(), none, none, stk, st), "tc_linear")
        p = L.WidePolicy()
        p.h2, p.w3, p.b3 = self.t2.data_ptr(), self._p(RP, o["w3"]), self._p(RP, o["b3"])
        p.rows, p.min_ac, p.max_ac = rows.data_ptr(), ag.min_ac.data_ptr(), ag.max_ac.data_ptr()
        p.eps, p.eps_out, p.xn, p.logp, p.save = L.ptr(eps_alpha), None, self.xq.data_ptr(), self.logp2.data_ptr(), None
        p.counters = ag.counters.data_ptr()
        p.M, p.O, p.A, p.out_dim, p.row_stride, p.ldn, p.src_off = M, O, ag.ac_dim, act.out_dim, rs, self.ldn, 0
        p.td3, p.smoothing, p.counter_idx, p.stream_id = 0, 0, L.CTR_PI, STREAM_ALPHA_EPS
        p.td3_std, p.td3_c, p.seed, p.agent = 0.0, 0.0, ag.hyper.seed, ag.base
        L.check(lib.b2rl_wide_policy_head(C.byref(p), stk, st), "wide_policy_head")
        L.check(lib.b2rl_wide_alpha_grad(self.logp2.data_ptr(), M, float(ag.hyper.targ_ent), ag.alpha_state.data_ptr(), stk, st),
                "wide_alpha_grad")


class WidePredictor:
    """``Agent.predict`` (agents/agent.py:172-181) for one learner on n observation rows, on the tensor cores: the
    observations are copied into a buffer whose rows TMA can address (pitch (O + 3) & ~3 floats; one memory-copy node, so
    they may sit in pinned host memory), then b2rl_tc_first -> b2rl_tc_linear -> b2rl_wide_actor_predict. Each actor weight
    is read once per 128 rows, where the row-group b2rl_actor_predict re-stages half of the actor per 8 rows; below 128
    rows most of the one tile is padding. The noise is b2rl_actor_predict's, number for number; the forward pass is 3xTF32
    (fp32-level) or TF32. Buffers are its own, sized for n. Enqueue-only (graph-capturable)."""

    def __init__(self, agent, n: int, precision: str = "3xtf32"):
        assert precision in ("3xtf32", "tf32")
        self.ag, self.n, self.x3 = agent, int(n), precision == "3xtf32"
        f32 = dict(dtype=torch.float32, device=agent.device)
        self.ldo = (agent.ob_dim + 3) & ~3
        self.x = torch.zeros(self.n, self.ldo, **f32)
        self.h1, self.h2 = torch.empty(self.n, 256, **f32), torch.empty(self.n, 256, **f32)
        # 3xTF32: the hidden layer's weight lo parts come from the learner's mirror, which its optimizer launches keep current
        self.wlo = agent.lo_mirror() if self.x3 else None

    def enqueue(self, obs_ptr: int, explore: bool, actions_ptr: int, eps: Optional[torch.Tensor] = None,
                eps_out: Optional[torch.Tensor] = None, draw: int = 2 ** 64 - 1, agent_hp: Optional[torch.Tensor] = None) -> None:
        """obs_ptr: [n][ob_dim] contiguous (device or pinned host); actions_ptr: [n][ac_dim] (device). draw as in
        b2rl_actor_predict: UINT64_MAX keys the noise on the critic step counter (inside a step graph)."""
        ag, lib, n = self.ag, self.ag._lib, self.n
        lay, st = ag.layout, ag._stream()
        act, o, RP = lay.actor, lay.actor.off, L.REGION_P
        ln = int(bool(ag.hps.layer_norm))
        p = lambda off: ag.arena.flat.data_ptr() + 4 * (RP * lay.region + off)
        L.check(lib.b2rl_copy_rows(self.x.data_ptr(), self.ldo, obs_ptr, ag.ob_dim, n, ag.ob_dim, st), "copy_rows")
        L.check(lib.b2rl_tc_first(self.x.data_ptr(), self.ldo, n, ag.ob_dim, p(o["w1t"]), p(o["b1"]), p(o["g1"]) if ln else None,
                                  p(o["be1"]) if ln else None, ln, self.h1.data_ptr(), None, None, int(self.x3), None, st), "tc_first")
        w = p(o["w2n"])
        wl = self.wlo.data_ptr() + (w - p(0)) if self.x3 else None
        L.check(lib.b2rl_tc_linear(self.h1.data_ptr(), 256, n, w, wl, p(o["b2"]), p(o["g2"]) if ln else None,
                                   p(o["be2"]) if ln else None, ln, 1, self.h2.data_ptr(), None, None, None, st), "tc_linear")
        q = L.WidePredict()
        q.h2, q.w3, q.b3 = self.h2.data_ptr(), p(o["w3"]), p(o["b3"])
        q.min_ac, q.max_ac = ag.min_ac.data_ptr(), ag.max_ac.data_ptr()
        q.eps, q.eps_out, q.actions = L.ptr(eps), L.ptr(eps_out), actions_ptr
        q.counters, q.agent_hp = ag.counters.data_ptr(), L.ptr(agent_hp)
        q.n, q.A, q.out_dim, q.mode, q.td3 = n, ag.ac_dim, act.out_dim, int(explore), int(ag.td3)
        q.explore_std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
        q.seed, q.draw, q.agent = ag.seed, int(draw), ag.agent_id
        L.check(lib.b2rl_wide_actor_predict(C.byref(q), st), "wide_actor_predict")
