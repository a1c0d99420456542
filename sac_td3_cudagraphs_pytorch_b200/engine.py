"""Whole learner iterations as CUDA graphs — the replacement for the reference's per-function
``CudaGraphModule`` wrapping (orchestrator.py:308-315) and its eager sample / Polyak calls
(orchestrator.py:338, :352).

One iteration of orchestrator.py:337-352 is: sample -> update_qnets -> (every
``actor_update_delay+1``-th iteration) ``actor_update_delay`` x update_actor on the same batch ->
update_targ_nets. Here that is ONE graph replay of 4 launches (critic-only iteration) or
4 + 4*delay launches (SAC; 3*delay for TD3): the sampler writes straight into the batch buffer the
update kernels read (no static-input copies), indices and noise come from Philox keyed on
device-side step counters (so replays need no host patching), and the Polyak average rides in the
Adam launch of the same parameters (legal: nothing reads the targets between the two, and
``target += polyak*(online_new - target)`` is the same arithmetic either way).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib as L
from .agents.agent import Agent
from .replay import Batch, ReplayBuffer
from .staging import StepStaging


class LearnerEngine:
    def __init__(self, agent: Agent, rb: Optional[ReplayBuffer] = None, batch_size: Optional[int] = None,
                 use_graphs: Optional[bool] = None, record_noise: bool = False, fused_opt: bool = False,
                 fused_sample: Optional[bool] = None):
        self.agent = agent
        self.rb = rb if rb is not None else agent.rb
        assert self.rb is not None and self.rb.storage is not None, "the replay buffer must hold data"
        self.B = int(batch_size or agent.hps.batch_size)
        self.use_graphs = bool(agent.hps.cudagraphs) if use_graphs is None else use_graphs
        # Adam + Polyak inside the weight-gradient kernel (b2rl_*_update_opt) instead of a launch of their own:
        # bitwise-equal results; measured on B200 at batch 256 it is ~1 us per iteration SLOWER (the optimizer's
        # dependent L2 round trips land on the tail of every gradient tile), so it is off by default
        self.fused_opt = bool(fused_opt)
        # the critic kernel draws the batch indices and reads the replay storage itself (and writes the batch rows out
        # for the kernels that follow) instead of a gather launch in front of it: same indices, bitwise-equal results,
        # one launch and one round trip of the batch through global memory less per iteration (TD3 Hopper 16.46 k ->
        # 16.96 k updates/s, SAC Humanoid 9.50 k -> 9.64 k: tools/bench_engine.py)
        self.fused_sample = True if fused_sample is None else bool(fused_sample)
        dev = agent.device
        self.rows = torch.zeros(self.B, agent.fmt.row_stride, dtype=torch.float32, device=dev)
        self.idx = torch.zeros(self.B, dtype=torch.int64, device=dev)
        delay = int(agent.hps.actor_update_delay)
        mk = (lambda: torch.zeros(self.B, agent.ac_dim, device=dev)) if record_noise else (lambda: None)
        # noise actually drawn by each step (parity tests replay a trajectory through the eager API)
        self.noise_q, self.noise_pi, self.noise_alpha = mk(), [mk() for _ in range(delay)], [mk() for _ in range(delay)]
        self.args_q = agent.update_args(self.rows, eps_out=self.noise_q,
                                        storage=self.rb.storage if self.fused_sample else None, idx_out=self.idx)
        self.args_pi = [agent.update_args(self.rows, eps_out=self.noise_pi[j], eps2_out=self.noise_alpha[j])
                        for j in range(delay)]
        self.graphs: dict[tuple, torch.cuda.CUDAGraph] = {}
        self._size_on_device = -1
        self._cursor_on_device = -1
        self.launches_per_variant: dict[tuple, int] = {}
        # end-to-end step (step_async / wait): pinned staging for the transitions and observations coming in, the log
        # block and the actions going out, two slots each (step parity) so one step may be in flight while the host
        # prepares the next
        self._stage = StepStaging(dev, (), agent.fmt.row_stride, agent.ob_dim, agent.ac_dim)
        self.host_out = self._stage.host_outs[0]
        self._keep: list = []
        self._side_stream = torch.cuda.Stream(device=dev)

    # -- what one iteration enqueues --------------------------------------------------------------
    def _enqueue(self, do_actor: bool, do_polyak: bool, args_q=None, before_last_adam=None) -> int:
        """before_last_adam: called right before the iteration's LAST Adam launch when nothing after that point writes
        the log block (i.e. not when SAC's temperature step follows): step graphs fork their publish node there."""
        ag, rb = self.agent, self.rb
        args_q = args_q or self.args_q
        st = ag._stream()
        n = 0
        if not self.fused_sample:
            L.check(ag._lib.b2rl_replay_sample_gather(
                rb.storage.data_ptr(), 0, 0, rb.fmt, self.B, 1, None, self.idx.data_ptr(), self.rows.data_ptr(),
                C.c_uint64(ag.seed), ag.counters.data_ptr(), L.CTR_Q, 0, ag.agent_id, st), "replay_sample_gather")
            n += 1
        delay = int(ag.hps.actor_update_delay) if do_actor else 0
        # TD3's target actor is averaged once per iteration, after the last actor update if there is one
        extra = ag.polyak_segs(critics=False, actor=True) if (ag.td3 and do_polyak and delay == 0) else []
        fused = ag.fuses_opt(self.fused_opt)  # (not with a lo mirror: only the stand-alone Adam launch writes it)
        hook = None if fused else before_last_adam
        ag.enqueue_critic_step(args_q, extra_segs=extra, polyak=do_polyak, fused_opt=fused,
                               before_adam=hook if delay == 0 else None)
        n += 2 if fused else 3
        for j in range(delay):
            ag.enqueue_actor_step(self.args_pi[j], polyak=ag.td3 and do_polyak and j == delay - 1,
                                  fused_opt=fused,
                                  before_adam=hook if (j == delay - 1 and not ag.autotune) else None)
            n += (5 if ag.hps.clip_norm > 0 else (2 if fused else 3)) + (1 if ag.autotune else 0)
        return n

    def _polyak_due(self) -> bool:
        ag = self.agent  # agents/agent.py:323-324, evaluated after the orchestrator bumped the counter
        return ag.td3 or ((ag.qnet_updates_so_far + 1) % ag.hps.crit_targ_update_freq == 0)

    def _sync_size(self) -> None:
        if self._size_on_device != len(self.rb):
            self._size_on_device = len(self.rb)
            self.agent.counters[L.CTR_SIZE] = self._size_on_device
        if self._cursor_on_device != self.rb._cursor:
            self._cursor_on_device = self.rb._cursor
            self.agent.counters[L.CTR_CURSOR] = self._cursor_on_device

    # -- the whole environment-facing step as ONE graph replay ---------------------------------------
    def host_rows(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [n, row_stride] for the transitions of the next step: fill it in place
        (replay.pack_rows(td, fmt, out=...)) and call step(i, n) / step_async(i, n). There are two slots (the parity
        of the step's sequence number; default: the next step's), so the buffer of step t may be filled while step
        t - 1 is still running — but only after wait() of step t - 2, which read from the same slot."""
        return self._stage.rows(n, slot)

    def host_obs(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [n, ob_dim] for the observations the policy acts on in the next step
        (step_async(..., n_obs=n)); two slots, like host_rows."""
        return self._stage.obs(n, slot)

    def wait_actions(self) -> "np.ndarray":
        """Actions of the last step launched with n_obs > 0 ([n_obs, A], a view of pinned host memory written by the
        device; valid until the step two launches later): polls the sequence number the step's policy part publishes
        — it runs FIRST in the graph, so the environments can step while the update of the same replay runs."""
        return self._stage.actions()

    def step_async(self, i: int, n_new: int = 0, n_obs: int = 0, explore: bool = True) -> int:
        """orchestrator.py:100-113 + :337-352 as ONE CUDA graph replay and no stream synchronisation: the replay
        write reads the n_new freshly collected transitions straight from pinned host memory (host_rows(n_new);
        cursor and fill count live on the device), then sample, critic update, delayed actor updates, Polyak,
        and a last kernel that writes the log block into pinned host memory and publishes a sequence number.
        Returns a ticket for wait(). At most two steps are in flight: a third first waits for the oldest (its
        staging slots are about to be reused). Needs graphs.
        n_obs > 0: the graph starts with the behaviour policy (Agent.predict, agents/agent.py:172-181, orchestrator.py
        :67-75) on the n_obs observations in host_obs(n_obs) — parameters as they are BEFORE this step's update, as in
        the reference loop — and publishes the actions to pinned host memory: wait_actions()."""
        ag, rb = self.agent, self.rb
        assert self.use_graphs, "step() is the graph path"
        slot = self._stage.begin()
        do_actor = (i % (ag.hps.actor_update_delay + 1) == 0)
        key = (do_actor, self._polyak_due(), int(n_new), slot, int(n_obs), bool(explore))
        self._sync_size()
        g = self.graphs.get(key)
        if g is None:
            g = self._capture_step(key)
        g.replay()
        if n_new:  # host mirror of the device-side cursor / fill count
            rb._cursor = (rb._cursor + n_new) % rb.capacity
            rb._size = min(rb.capacity, rb._size + n_new)
            self._cursor_on_device, self._size_on_device = rb._cursor, rb._size
        ag.qnet_updates_so_far += 1
        if do_actor:
            ag.actor_updates_so_far += int(ag.hps.actor_update_delay)
        return self._stage.launched(n_obs, slot)

    def wait(self, ticket: int, as_numpy: bool = False):
        """Poll the sequence number the step's last kernel publishes; returns that step's pinned log block
        (_lib.OUT_* indices; a torch tensor, or its numpy view), valid until the step two tickets later is launched."""
        return self._stage.wait(ticket, as_numpy)

    def step(self, i: int, n_new: int = 0, n_obs: int = 0, explore: bool = True) -> torch.Tensor:
        """step_async + wait: the loop of a trainer that reads the losses of every step before the next one."""
        return self.wait(self.step_async(i, n_new, n_obs, explore))

    def _capture_step(self, key) -> torch.cuda.CUDAGraph:
        ag, rb, stage = self.agent, self.rb, self._stage
        do_actor, do_polyak, n_new, slot, n_obs, explore = key
        new_rows = stage.rows(n_new, slot) if n_new else None
        if n_obs:
            obs = stage.obs(n_obs, slot)
            pa = L.UpdateArgs()
            pa.hp, pa.fmt, pa.actor = ag._hyper, ag.fmt, ag.layout.actor.c_struct()
            pa.arena, pa.region_stride, pa.agent_base = ag.arena.flat.data_ptr(), ag.layout.region, ag.agent_id
            pa.min_ac, pa.max_ac, pa.counters = ag.min_ac.data_ptr(), ag.max_ac.data_ptr(), ag.counters.data_ptr()
            self._keep.append(pa)
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(ag.device)
        with torch.cuda.graph(g):
            n = 0
            if n_obs:  # the policy first: the environments get their actions while the update runs
                std = float(ag.hps.actor_noise_std) if ag.td3 else 0.0
                L.check(ag._lib.b2rl_actor_predict(C.byref(pa), obs.data_ptr(), n_obs, int(explore), std,
                                                   C.c_uint64(2 ** 64 - 1), stage.device_actions(n_obs).data_ptr(), ag._stream()),
                        "actor_predict")
                stage.publish_actions(ag._lib, n_obs, slot, ag._stream())
                n += 2
            args_q = None
            if n_new and self.fused_sample and not ag.fuses_opt(self.fused_opt):
                # the replay write rides in the critic step too (b2rl_update_args_t.new_rows): the kernel reads the pinned
                # rows itself (UVA), no separate write launch
                args_q = ag.update_args(self.rows, eps_out=self.noise_q, storage=rb.storage, idx_out=self.idx,
                                        new_rows=new_rows, n_new=n_new)
                self._keep.append(args_q)
            elif n_new:  # pinned host memory is device-addressable (UVA): the write kernel is the host->device copy
                L.check(ag._lib.b2rl_replay_extend_dev(rb.storage.data_ptr(), rb.capacity, rb.fmt,
                                                       new_rows.data_ptr(), n_new, ag.counters.data_ptr(),
                                                       ag._stream()), "replay_extend_dev")
                n += 1
            # The log block is final before the iteration's last Adam launch (unless SAC's temperature step follows):
            # the publish node forks off there and runs beside Adam instead of after it.
            joined = []

            def publish():
                stage.publish_logs(ag._lib, ag.out, slot, ag._stream())

            def fork_publish():
                main, ev = torch.cuda.current_stream(ag.device), torch.cuda.Event()
                ev.record(main)
                self._side_stream.wait_event(ev)
                with torch.cuda.stream(self._side_stream):
                    publish()
                    done = torch.cuda.Event()
                    done.record(self._side_stream)
                joined.append(done)

            n += self._enqueue(do_actor, do_polyak, args_q, before_last_adam=fork_publish)
            if joined:
                torch.cuda.current_stream(ag.device).wait_event(joined[0])
            else:
                publish()
            n += 1
        self.launches_per_variant[key] = n
        self.graphs[key] = g
        return g

    def iteration(self, i: int) -> None:
        """One learner iteration (orchestrator.py:337-352) — enqueue only, nothing is read back."""
        ag = self.agent
        do_actor = (i % (ag.hps.actor_update_delay + 1) == 0)
        key = (do_actor, self._polyak_due())
        self._sync_size()
        if not self.use_graphs:
            self.launches_per_variant[key] = self._enqueue(*key)
        else:
            g = self.graphs.get(key)
            if g is None:
                g = self._capture(key)
            g.replay()
        ag.qnet_updates_so_far += 1
        if do_actor:
            ag.actor_updates_so_far += int(ag.hps.actor_update_delay)

    def _capture(self, key) -> torch.cuda.CUDAGraph:
        """Capture the variant. Capture itself executes nothing, so learner state is untouched."""
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(self.agent.device)
        with torch.cuda.graph(g):
            self.launches_per_variant[key] = self._enqueue(*key)
        self.graphs[key] = g
        return g

    def launches(self, i: int) -> int:
        key = (i % (self.agent.hps.actor_update_delay + 1) == 0, self._polyak_due())
        return self.launches_per_variant.get(key, 0)

    def logs(self) -> dict[str, torch.Tensor]:
        """The reference's log keys (agents/agent.py:238-242, :288-318) as views of the device-side
        output block — no clone, no sync; read them when you log."""
        ag, o = self.agent, self.agent.out
        d = {"loss/qf_loss": o[L.OUT_QF_LOSS], "loss/actor_loss": o[L.OUT_ACTOR_LOSS]}
        if not ag.td3:
            d["vitals/alpha"] = o[L.OUT_ALPHA]
            if ag.autotune:
                d["loss/alpha_loss"] = o[L.OUT_ALPHA_LOSS]
        return d

    def last_batch(self) -> Batch:
        return Batch(self.rows, self.agent.fmt, self.idx)
