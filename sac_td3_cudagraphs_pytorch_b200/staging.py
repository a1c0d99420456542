"""Host side of an environment-facing step graph (LearnerEngine.step_async, Population.step_async): pinned staging
buffers for the transitions and observations going in, pinned log blocks and actions coming out, and the sequence
numbers the device publishes after each (b2rl_publish_logs) so the host polls memory instead of synchronising a stream.

Every buffer has two slots, chosen by the parity of the step's sequence number, so the host may fill the inputs of
step t while step t - 1 is still running; at most two steps are in flight. `lead` is the leading shape of every staged
array: () for one learner, (N,) for a population of N agents.
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Optional

import numpy as np
import torch

from . import _lib as L


class StepStaging:
    def __init__(self, device, lead: tuple, row_stride: int, ob_dim: int, ac_dim: int):
        self.device, self.lead = torch.device(device), tuple(lead)
        self.n_agents = int(np.prod(self.lead)) if self.lead else 1
        self.row_stride, self.ob_dim, self.ac_dim = int(row_stride), int(ob_dim), int(ac_dim)
        self._h_new: dict[tuple, torch.Tensor] = {}
        self._h_obs: dict[tuple, torch.Tensor] = {}
        self._h_act: dict[tuple, torch.Tensor] = {}
        self._d_act: dict[int, torch.Tensor] = {}
        self.host_outs = [torch.zeros(*self.lead, 8, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._host_outs_np = [t.numpy() for t in self.host_outs]
        self._host_act_seq = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._host_act_seq_np = self._host_act_seq.numpy()
        self._act_seq_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._act_seq, self._act_last = 0, None
        self._host_seq = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._host_seq_np = self._host_seq.numpy()  # (a view: polled without going through torch)
        self._seq_dev = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.seq = 0  # steps launched
        self.waited = 0  # highest ticket waited for

    def slot(self, slot: Optional[int] = None) -> int:
        """The staging slot of the next step (default) or the given one."""
        return (self.seq & 1) if slot is None else int(slot) & 1

    def rows(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned [*lead, n, row_stride] transitions of a step."""
        key = (int(n), self.slot(slot))
        if key not in self._h_new:
            self._h_new[key] = torch.zeros(*self.lead, n, self.row_stride, dtype=torch.float32).pin_memory()
        return self._h_new[key]

    def obs(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned [*lead, n, ob_dim] observations the step's policy acts on."""
        key = (int(n), self.slot(slot))
        if key not in self._h_obs:
            self._h_obs[key] = torch.zeros(*self.lead, n, self.ob_dim, dtype=torch.float32).pin_memory()
            blocks = (self.n_agents * n * self.ac_dim + 7) // 8  # b2rl_publish_logs copies blocks of 8 floats
            self._h_act[key] = torch.zeros(blocks * 8, dtype=torch.float32).pin_memory()
            if n not in self._d_act:
                self._d_act[n] = torch.zeros(blocks * 8, dtype=torch.float32, device=self.device)
        return self._h_obs[key]

    def device_actions(self, n: int) -> torch.Tensor:
        """The device buffer the step's policy writes (then published to the pinned slot)."""
        return self._d_act[n]

    def publish_actions(self, lib, n: int, slot: int, stream: int) -> None:
        d = self._d_act[n]
        L.check(lib.b2rl_publish_logs(d.data_ptr(), d.numel() // 8, self._h_act[(n, slot)].data_ptr(), self._act_seq_dev.data_ptr(),
                                      self._host_act_seq.data_ptr(), stream), "publish actions")

    def publish_logs(self, lib, out: torch.Tensor, slot: int, stream: int) -> None:
        L.check(lib.b2rl_publish_logs(out.data_ptr(), self.n_agents, self.host_outs[slot].data_ptr(), self._seq_dev.data_ptr(),
                                      self._host_seq.data_ptr(), stream), "publish_logs")

    def begin(self) -> int:
        """Slot of the step about to be launched; with two steps in flight, first waits for the older one (its staging
        slots are about to be reused)."""
        if self.seq - self.waited >= 2:
            self.wait(self.seq - 1)
        return self.seq & 1

    def launched(self, n_obs: int, slot: int) -> int:
        """Record a launched step; returns its ticket for wait()."""
        self.seq += 1
        if n_obs:
            self._act_seq += 1
            self._act_last = (int(n_obs), slot, self._act_seq)
        return self.seq

    def wait(self, ticket: int, as_numpy: bool = False):
        """Poll the sequence number the step's last kernel publishes; returns that step's pinned log block [*lead, 8]
        (_lib.OUT_* indices; a torch tensor, or its numpy view), valid until the step two tickets later is launched."""
        self.poll(self._host_seq_np, ticket, "the step's log block")  # written after the log block (system-scope fence)
        self.waited = max(self.waited, int(ticket))
        return (self._host_outs_np if as_numpy else self.host_outs)[(ticket - 1) & 1]

    def actions(self) -> "np.ndarray":
        """Actions [*lead, n_obs, A] of the last step launched with n_obs > 0 (a view of pinned host memory written by
        the device; valid until the step two launches later)."""
        if self._act_last is None:
            raise L.B2rlError("no step with n_obs > 0 has been launched")
        n, slot, want = self._act_last
        self.poll(self._host_act_seq_np, want, "the policy's actions")
        return self._h_act[(n, slot)].numpy()[: self.n_agents * n * self.ac_dim].reshape(*self.lead, n, self.ac_dim)

    def poll(self, seq, want: int, what: str, timeout_s: float = 30.0) -> None:
        """Spin on a pinned sequence number the device publishes. Every 4096 empty polls the stream is queried: a step
        that has FINISHED without publishing (a faulted replay: the publish kernel never ran) or a deadline miss raises
        instead of hanging the host."""
        spins, t0 = 0, None
        while seq[0] < want:
            spins += 1
            if spins & 0xFFF:
                continue
            t0 = t0 or time.monotonic()
            done = torch.cuda.current_stream(self.device).query()  # raises on a sticky CUDA error
            if done and seq[0] < want:
                raise L.B2rlError(f"the stream drained but {what} was never published (sequence {int(seq[0])} < {want})")
            if time.monotonic() - t0 > timeout_s:
                raise L.B2rlError(f"timed out after {timeout_s:.0f} s waiting for {what} (sequence {int(seq[0])} < {want})")
