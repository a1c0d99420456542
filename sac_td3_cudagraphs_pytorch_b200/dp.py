"""Large-batch data-parallel learner (BASELINE.json config 5): W replicas of one agent, each with its own
replay buffer and its own batch; gradients of the mean loss are summed over ranks with one
`all_reduce` per optimizer step on the flat gradient span of the arena (NCCL over NVLink on GPUs) and the
`1/W` is folded into the Adam kernel (`grad_scale`). The reference has no counterpart (no
torch.distributed anywhere, SURVEY §2.2); the parity oracle is a single rank run on the concatenation of
the W local batches (mean of equal-sized means = global mean).

Replicas stay bit-identical: every rank applies the same reduced gradient with the same arithmetic. The
natural-layout shadows (`w2n`) never see a gradient of their own — a ring all-reduce may sum two positions of the
buffer in different orders — the Adam launch steps `w2t` and writes the result to both layouts (adam.cu).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.distributed as dist

from . import _lib as L
from .arena import Arena, ArenaLayout
from .staging import StepStaging


class GradComm:
    """Sum-all-reduce over a torch.distributed group (NCCL on GPUs, gloo in the CPU tests)."""

    def __init__(self, group=None):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0

    def all_reduce_sum(self, t: torch.Tensor) -> None:
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)


def reduce_grad_span(arena: Arena, layout: ArenaLayout, comm: GradComm, which: str, agent: int = 0) -> None:
    """All-reduce the gradients (region 4) of the critics or of the actor, then rebuild the w2n shadows."""
    if comm.world == 1:  # nothing to reduce, and the weight-gradient kernels wrote the shadows themselves
        return
    nets = layout.critic if which == "critic" else [layout.actor]
    g = arena.flat[agent, L.REGION_G]
    # one contiguous bucket (a shadow's gradient slot in between rides along unused: the Adam launch derives the w2n
    # shadows from the reduced w2t gradient through its transposing tiles, so replicas stay bit-identical with no copy)
    comm.all_reduce_sum(g[nets[0].begin:nets[-1].core_end])


class DataParallelLearner:
    """One rank of the data-parallel learner. `agent` must be constructed identically on every rank (same
    torch seed => same initial parameters) except `agent_id=rank`, which keys its index/noise draws."""

    def __init__(self, agent, rb, batch_size: int, comm: Optional[GradComm] = None, wide: Optional[str] = None,
                 graphs: Optional[bool] = None, policy: Optional[str] = None):
        """wide: None = row-group kernels; "3xtf32" / "tf32" = the critic step on the layer-by-layer tensor-core path
        (wide.WideCritic), which is what a batch of tens of thousands wants.
        policy: the behaviour policy of step_async(n_obs > 0). "row" (default) = b2rl_actor_predict (2-CTA clusters on
        8-row tiles); "wide" = wide.WidePredictor (tensor cores, the learner's precision; needs a wide learner; below 128
        observation rows it computes one mostly empty tile). Measured on a B200, Hopper, 3xTF32, 256 to 16 384 observation
        rows, the row kernel was the faster at every size (profiles/r3_dp_step.json, DESIGN §5), so it is the default."""
        self.agent, self.rb, self.B = agent, rb, int(batch_size)
        self.policy = policy or "row"
        if self.policy not in ("row", "wide") or (self.policy == "wide" and not wide):
            raise L.B2rlError(f"policy must be 'row' or, with a wide learner, 'wide' (got {policy!r}, wide={wide!r})")
        self.precision = wide
        self.wide = self.wide_actor = None
        if wide:
            from .wide import WideActor, WideCritic
            self.wide = WideCritic(agent, self.B, wide)
            if not agent.hps.clip_norm > 0:  # (the wide actor step has no gradient clipping)
                self.wide_actor = WideActor(agent, self.B, wide)
        self.comm = comm or GradComm()
        dev = agent.device
        self.rows = torch.zeros(self.B, agent.fmt.row_stride, dtype=torch.float32, device=dev)
        self.idx = torch.zeros(self.B, dtype=torch.int64, device=dev)
        self.launches = 0
        # One CUDA graph per iteration variant (actor updates? Polyak?) when the batch is sampled on the device: the wide
        # path is ~100 launches per iteration, ~0.9 ms of host time to enqueue — all of a batch-16 384 iteration
        # (tools/dp_cpu_time.py). With W > 1 the NCCL all-reduces are captured INSIDE the iteration graph (NCCL collectives
        # are stream-capturable; every rank replays the same sequence), so the multi-rank iteration is one graph launch
        # too; other backends (gloo in the CPU-side tests) stay eager.
        capturable = self.comm.world == 1 or (dist.is_initialized() and dist.get_backend(self.comm.group) == "nccl")
        self.graphs = (capturable and rb is not None and bool(agent.hps.cudagraphs)) if graphs is None else bool(graphs)
        self._graphs: dict[tuple, torch.cuda.CUDAGraph] = {}
        self._size_on_device = -1
        self._cursor_on_device = -1
        self._warm: set = set()
        # environment-facing step (step_async / wait), as LearnerEngine's: pinned staging in and out, two slots each
        self._stage = StepStaging(dev, (), agent.fmt.row_stride, agent.ob_dim, agent.ac_dim)
        self._step_graphs: dict[tuple, torch.cuda.CUDAGraph] = {}
        self._predictors: dict[int, object] = {}
        self._keep: list = []

    def _seg(self, begin, end, lr, polyak, counter, clip=False):
        return L.Seg(begin, end, lr, 1, int(polyak), counter, 1.0 / self.comm.world, int(clip))

    def iteration(self, i: int, rows: Optional[torch.Tensor] = None, eps_q=None, eps_pi=None, eps_alpha=None) -> None:
        """One iteration of orchestrator.py:337-352 with gradient averaging over ranks. `rows` / `eps_*`
        inject this rank's batch and noise (parity tests); default: device-side sampling."""
        ag, lib, lay, h, W = self.agent, self.agent._lib, self.agent.layout, self.agent.hps, self.comm.world
        do_actor = (i % (h.actor_update_delay + 1) == 0)
        do_polyak = ag.td3 or ((ag.qnet_updates_so_far + 1) % h.crit_targ_update_freq == 0)
        if rows is None and self._size_on_device != len(self.rb):
            self._size_on_device = len(self.rb)
            ag.counters[L.CTR_SIZE] = self._size_on_device
        if self.graphs and rows is None and eps_q is None and eps_pi is None and eps_alpha is None:
            key = (do_actor, do_polyak)
            g = self._graphs.get(key)
            if g is None:  # first occurrence of the variant runs eagerly (lazy allocations), the second is captured
                if key not in self._warm:
                    self._warm.add(key)
                else:
                    g = torch.cuda.CUDAGraph()
                    torch.cuda.synchronize(ag.device)
                    with torch.cuda.graph(g):
                        self._enqueue(do_actor, do_polyak, None, None, None, None)
                    self._graphs[key] = g  # (capture does not execute: the replay below is this iteration)
            if g is not None:
                g.replay()
                return self._count(do_actor)
        self._enqueue(do_actor, do_polyak, rows, eps_q, eps_pi, eps_alpha)
        self._count(do_actor)

    def _count(self, do_actor: bool) -> None:
        ag = self.agent
        ag.qnet_updates_so_far += 1
        if do_actor:
            ag.actor_updates_so_far += int(ag.hps.actor_update_delay)

    def _enqueue(self, do_actor, do_polyak, rows, eps_q, eps_pi, eps_alpha) -> None:
        ag, lib, lay, h, W = self.agent, self.agent._lib, self.agent.layout, self.agent.hps, self.comm.world
        st = ag._stream()
        if rows is None:
            L.check(lib.b2rl_replay_sample_gather(
                self.rb.storage.data_ptr(), 0, 0, self.rb.fmt, self.B, 1, None, self.idx.data_ptr(),
                self.rows.data_ptr(), C.c_uint64(ag.seed), ag.counters.data_ptr(), L.CTR_Q, 0, ag.agent_id, st),
                "replay_sample_gather")
            rows = self.rows
        delay = int(h.actor_update_delay) if do_actor else 0

        if self.wide is not None:
            self.wide.update_qnets(rows, eps=ag._noise(eps_q, rows), adam=False)
        else:
            args = ag.update_args(rows, eps=ag._noise(eps_q, rows))
            fn = lib.b2rl_critic_update_td3 if ag.td3 else lib.b2rl_critic_update_sac
            L.check(fn(C.byref(args), st), "critic_update")
        reduce_grad_span(ag.arena, lay, self.comm, "critic")
        segs = [self._seg(lay.critic[0].begin, lay.critic[1].end, float(h.qnets_lr), do_polyak, L.CTR_Q)]
        if ag.td3 and do_polyak and delay == 0:
            segs.append(L.Seg(lay.actor.begin, lay.actor.end, 0.0, 0, 1, 0, 1.0, 0))
        ag._launch_adam(segs)
        for j in range(delay):
            e1 = None if eps_pi is None else eps_pi[j]
            e2 = None if eps_alpha is None else eps_alpha[j]
            args = ag.update_args(rows, eps=ag._noise(e1, rows), eps2=ag._noise(e2, rows))
            if self.wide_actor is not None:
                self.wide_actor.update_actor(rows, eps=ag._noise(e1, rows), adam=False)
            else:
                fn = lib.b2rl_actor_update_td3 if ag.td3 else lib.b2rl_actor_update_sac
                L.check(fn(C.byref(args), st), "actor_update")
            reduce_grad_span(ag.arena, lay, self.comm, "actor")
            clip = h.clip_norm > 0
            if clip:  # clip_grad_norm_ acts on the averaged gradient: sum of squares AFTER the all-reduce
                L.check(lib.b2rl_grad_sumsq(ag.arena.flat.data_ptr(), lay.region, ag.arena.agent_stride,
                                            lay.actor.begin, lay.actor.core_end, 1, ag._sumsq.data_ptr(),
                                            ag._sumsq_scratch.data_ptr(), st), "grad_sumsq")
            ag._launch_adam([self._seg(lay.actor.begin, lay.actor.end, float(h.actor_lr),
                                       ag.td3 and do_polyak and j == delay - 1, L.CTR_PI, clip)])
            if ag.autotune:
                if self.wide_actor is not None:
                    self.wide_actor.alpha_grad(rows, ag._noise(e2, rows))
                else:
                    L.check(lib.b2rl_alpha_update(C.byref(args), 0.0, st), "alpha_update (gradient only)")
                self.comm.all_reduce_sum(ag._alpha_state[1:2])
                L.check(lib.b2rl_alpha_adam(ag._alpha_state.data_ptr(), ag.counters.data_ptr(), 1,
                                            float(h.log_alpha_lr), 1.0 / W, ag.out.data_ptr(), st), "alpha_adam")

    # -- the whole environment-facing step as ONE graph replay (LearnerEngine.step_async for this learner) -------------------
    def host_rows(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [n, row_stride] for this rank's transitions of the next step (replay.pack_rows(td, fmt,
        out=...)); two slots, as LearnerEngine.host_rows: fill the next step's while the previous one runs."""
        return self._stage.rows(n, slot)

    def host_obs(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [n, ob_dim] for the observations the next step's policy acts on; two slots."""
        return self._stage.obs(n, slot)

    def wait_actions(self) -> "np.ndarray":
        """Actions [n_obs, A] of the last step launched with n_obs > 0 (pinned host memory, valid until the step two
        launches later). The policy runs first in the step graph, so the environments can step while the update runs."""
        return self._stage.actions()

    def wait(self, ticket: int, as_numpy: bool = False):
        """This rank's log block of the step with that ticket (_lib.OUT_*), valid until the step two tickets later."""
        return self._stage.wait(ticket, as_numpy)

    def step(self, i: int, n_new: int = 0, n_obs: int = 0, explore: bool = True):
        """step_async + wait."""
        return self.wait(self.step_async(i, n_new, n_obs, explore))

    def step_async(self, i: int, n_new: int = 0, n_obs: int = 0, explore: bool = True) -> int:
        """orchestrator.py:67-113 + :337-352 for this rank as ONE CUDA graph replay and no stream synchronisation: the
        behaviour policy on the n_obs observations in host_obs(n_obs) with the parameters as they are BEFORE this step's
        update (as in the reference loop), its actions published to pinned memory (wait_actions); the n_new transitions
        in host_rows(n_new) appended to the replay (cursor and fill count live on the device); iteration(i) — with W > 1
        its NCCL all-reduces inside the graph, every rank replaying the same sequence; the log block published (wait).
        Returns a ticket. At most two steps are in flight: a third first waits for the oldest. Needs graphs."""
        ag, rb = self.agent, self.rb
        if not self.graphs or rb is None or rb.storage is None:
            raise L.B2rlError("step_async needs iteration graphs (NCCL or one rank, cudagraphs on) and a replay buffer holding data")
        if not (isinstance(n_new, int) and isinstance(n_obs, int)) or n_new < 0 or n_obs < 0:
            raise L.B2rlError(f"step_async: n_new and n_obs must be ints >= 0 (got {n_new!r}, {n_obs!r})")
        if n_new > rb.capacity:
            raise L.B2rlError(f"step_async: n_new {n_new} exceeds the replay capacity {rb.capacity}")
        do_actor = (i % (ag.hps.actor_update_delay + 1) == 0)
        do_polyak = ag.td3 or ((ag.qnet_updates_so_far + 1) % ag.hps.crit_targ_update_freq == 0)
        slot = self._stage.begin()
        key = (do_actor, do_polyak, n_new, slot, n_obs, bool(explore))
        if self._size_on_device != len(rb):
            self._size_on_device = len(rb)
            ag.counters[L.CTR_SIZE] = self._size_on_device
        if self._cursor_on_device != rb._cursor:
            self._cursor_on_device = rb._cursor
            ag.counters[L.CTR_CURSOR] = self._cursor_on_device
        g = self._step_graphs.get(key)
        if g is None and key not in self._warm:  # first occurrence eagerly (lazy allocations, NCCL set-up), then captured
            self._warm.add(key)
            self._enqueue_step(key)
        else:
            if g is None:
                g = self._step_graphs[key] = torch.cuda.CUDAGraph()
                torch.cuda.synchronize(ag.device)
                with torch.cuda.graph(g):
                    self._enqueue_step(key)
            g.replay()
        if n_new:  # host mirror of the device-side cursor / fill count: iteration() uploads no stale size over them
            rb._cursor = (rb._cursor + n_new) % rb.capacity
            rb._size = min(rb.capacity, rb._size + n_new)
            self._cursor_on_device, self._size_on_device = rb._cursor, rb._size
        self._count(do_actor)
        return self._stage.launched(n_obs, slot)

    def _enqueue_step(self, key) -> None:
        ag, rb, stage = self.agent, self.rb, self._stage
        do_actor, do_polyak, n_new, slot, n_obs, explore = key
        st = ag._stream()
        if n_obs:
            obs, act = stage.obs(n_obs, slot), stage.device_actions(n_obs)
            if self.policy == "wide":
                pol = self._predictors.get(n_obs)
                if pol is None:
                    from .wide import WidePredictor
                    pol = self._predictors[n_obs] = WidePredictor(ag, n_obs, self.precision)
                pol.enqueue(obs.data_ptr(), explore, act.data_ptr())
            else:
                pa = L.UpdateArgs()
                pa.hp, pa.fmt, pa.actor = ag._hyper, ag.fmt, ag.layout.actor.c_struct()
                pa.arena, pa.region_stride, pa.agent_base = ag.arena.flat.data_ptr(), ag.layout.region, ag.agent_id
                pa.min_ac, pa.max_ac, pa.counters = ag.min_ac.data_ptr(), ag.max_ac.data_ptr(), ag.counters.data_ptr()
                self._keep.append(pa)
                std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
                L.check(ag._lib.b2rl_actor_predict(C.byref(pa), obs.data_ptr(), n_obs, int(explore), std, C.c_uint64(2 ** 64 - 1),
                                                   act.data_ptr(), st), "actor_predict")
            stage.publish_actions(ag._lib, n_obs, slot, st)
        if n_new:  # pinned host memory is device-addressable (UVA): the write kernel is the host->device copy
            L.check(ag._lib.b2rl_replay_extend_dev(rb.storage.data_ptr(), rb.capacity, rb.fmt, stage.rows(n_new, slot).data_ptr(),
                                                   n_new, ag.counters.data_ptr(), st), "replay_extend_dev")
        self._enqueue(do_actor, do_polyak, None, None, None, None)
        stage.publish_logs(ag._lib, ag.out, slot, st)
