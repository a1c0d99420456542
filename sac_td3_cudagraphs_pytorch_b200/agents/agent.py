"""``Agent`` — the learner object orchestrator.py drives, with the reference's call surface
(agents/agent.py:24-331) on top of the B200-native update path:

    reference (torch ops, ~330 kernels / full update)        here (libb2rl.so, sm_100a)
    -------------------------------------------------        -----------------------------------
    update_qnets   agents/agent.py:183-242                   critic.cu + wgrad.cu + adam.cu   (3 launches)
    update_actor   agents/agent.py:244-318                   actor.cu + wgrad.cu + adam.cu [+ alpha] (3-4)
    update_targ_nets agents/agent.py:320-331                 adam.cu polyak-only segments     (1)
    predict        agents/agent.py:172-181                   actor.cu predict_kernel          (1)

All learner state lives in one flat fp32 arena (arena.py); ``actor``, ``qnet1``, ``qnet2``,
``qnet_params``, ``qnet_target`` ... are views of it with the reference's names and shapes.
The update needs a CUDA device and the compiled library: there is no CPU or torch fallback.
Every launch goes to the current torch stream and is CUDA-graph capturable; engine.py captures
whole learner iterations.
"""
from __future__ import annotations

import ctypes as C
import math
from pathlib import Path
from typing import Any, Mapping, Optional

import numpy as np
import torch

from .. import _lib as L
from ..arena import Arena, NetLayout, TENSOR_NAMES, make_layout, set_shadow_pairs
from ..hps import hp_get
from ..replay import Batch, pack_rows, row_format
from .nets import Actor, Critic, TanhGaussActor, log_module_info

HID_DIMS = (256, 256)  # agents/agent.py:56,101


class ArenaAdam:
    """torch.optim.Adam-shaped handle on optimizer state that lives in arena regions 2/3
    (betas (0.9, 0.999), eps 1e-8, no weight decay: agents/agent.py:115-139)."""

    def __init__(self, agent: "Agent", params: dict[str, torch.Tensor], m: dict, v: dict, lr: float,
                 counter: int, spans: list[tuple[int, int]]):
        self._agent, self._params, self._m, self._v = agent, params, m, v
        self.counter, self.spans = counter, spans
        self.param_groups = [dict(lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0, amsgrad=False,
                                  maximize=False, capturable=True, params=list(range(len(params))))]

    @property
    def lr(self) -> float:
        return float(self.param_groups[0]["lr"])

    @property
    def step_count(self) -> int:
        return int(self._agent.counters[self.counter].item())

    def zero_grad(self, set_to_none: bool = True) -> None:
        """No-op: the backward kernels overwrite every gradient element (nothing accumulates)."""

    def step(self) -> None:
        """Apply Adam to the gradients currently in region 4 (advances the step count first). Like
        torch.optim.Adam.step() it does NOT clip: gradient clipping (hps.clip_norm) is part of Agent.update_actor."""
        ag = self._agent
        st = ag._stream()
        if not self.spans:  # the temperature: a scalar whose gradient sits in its state block (slot 1)
            L.check(ag._lib.b2rl_alpha_adam(ag._alpha_state.data_ptr(), ag.counters.data_ptr(), 1, self.lr, 1.0,
                                            ag.out.data_ptr(), st), "alpha_adam")  # (bumps counters[ALPHA] itself)
            return
        L.check(ag._lib.b2rl_bump_counter(ag.counters.data_ptr(), self.counter, 1, st), "bump_counter")
        ag._launch_adam([ag._seg(b, e, self.lr, adam=True, polyak=False, counter=self.counter) for b, e in self.spans])

    def state_dict(self) -> dict:
        step = torch.tensor(float(self.step_count))
        state = {i: {"step": step.clone(), "exp_avg": self._m[n].detach().clone(),
                     "exp_avg_sq": self._v[n].detach().clone()} for i, n in enumerate(self._params)}
        return {"state": state if self.step_count > 0 else {}, "param_groups": [dict(g) for g in self.param_groups]}

    @torch.no_grad()
    def load_state_dict(self, sd: dict) -> None:
        for i, n in enumerate(self._params):
            if i in sd["state"]:
                self._m[n].copy_(sd["state"][i]["exp_avg"])
                self._v[n].copy_(sd["state"][i]["exp_avg_sq"])
                self._agent.counters[self.counter] = int(sd["state"][i]["step"])
        self.param_groups[0]["lr"] = sd["param_groups"][0]["lr"]
        self._agent.arena.sync_shadows((L.REGION_M, L.REGION_V))


def checkpoint_path(path, sfx: Optional[str], timesteps_so_far: int) -> Path:
    """File name of a checkpoint in directory `path` (agents/agent.py:337-341)."""
    fname = f"ckpt_{sfx}" if sfx is not None else f".ckpt_{timesteps_so_far}ts"
    return Path(path) / f"{fname}.pth"


def checkpoint_dict(hps, timesteps_so_far: int, actor, qnet1, qnet2, actor_optimizer: ArenaAdam, q_optimizer: ArenaAdam,
                    actor_target: Mapping[str, torch.Tensor], qnet_target: Mapping[str, torch.Tensor],
                    log_alpha: Optional[torch.Tensor] = None, alpha_optimizer: Optional[ArenaAdam] = None) -> dict:
    """The dict Agent.save writes and Agent.load_from_disk reads: the reference's layout (agents/agent.py:343-352) plus
    targets and temperature. actor / qnet1 / qnet2 are nets.py modules (their state_dicts), targets map the reference's
    names to tensors ([2, ...] for the critics), log_alpha / alpha_optimizer are SAC's (the optimizer with autotune)."""
    clone = lambda sd: {k: v.detach().clone().contiguous() for k, v in sd.items()}
    ckpt = {
        "hps": dict(hps) if isinstance(hps, Mapping) else hps,
        "timesteps_so_far": timesteps_so_far,
        "actor": clone(actor.state_dict()),
        "qnet1": clone(qnet1.state_dict()),
        "qnet2": clone(qnet2.state_dict()),
        "actor_optimizer": actor_optimizer.state_dict(),
        "q_optimizer": q_optimizer.state_dict(),
        "actor_target": clone(actor_target),
        "qnet_target": clone(qnet_target),
    }
    if log_alpha is not None:
        ckpt["log_alpha"] = log_alpha.detach().clone()
    if alpha_optimizer is not None:
        ckpt["alpha_optimizer"] = alpha_optimizer.state_dict()
    return ckpt


class Agent:

    def __init__(self, net_shapes: dict[str, tuple[int, ...]], min_ac: np.ndarray, max_ac: np.ndarray,
                 device: torch.device, hps: Any, rb: Optional[Any] = None, seed: int = 0, agent_id: int = 0):
        ob_shape, ac_shape = net_shapes["ob_shape"], net_shapes["ac_shape"]
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.B2rlError("the B200-native Agent needs a CUDA device (there is no CPU path)")
        self._lib = L.load()
        L.init_device(self.device)
        self.ob_dim, self.ac_dim = int(ob_shape[-1]), int(ac_shape[-1])
        self.min_ac = torch.tensor(min_ac, dtype=torch.float, device=self.device)
        self.max_ac = torch.tensor(max_ac, dtype=torch.float, device=self.device)
        self.hps = hps
        self.td3 = bool(hps.prefer_td3_over_sac)
        self.seed = int(seed)
        self.agent_id = int(agent_id)  # global learner id (Philox key); a Population member g has agent_id base+g

        self.timesteps_so_far = 0
        self.actor_updates_so_far = 0
        self.qnet_updates_so_far = 0
        self.best_eval_ep_ret = -float("inf")  # updated by the training loop (orchestrator.py:376-379)

        assert hps.segment_len <= hps.batch_size
        self.rb = rb
        self.fmt = row_format(self.ob_dim, self.ac_dim)
        self.batch_size = int(hps.batch_size)

        # ---- arena and networks
        ln = bool(hps.layer_norm)
        self.layout = make_layout(self.ob_dim, self.ac_dim, self.td3, ln)
        self.arena = Arena(self.layout, self.device)
        ar, lay = self.arena, self.layout

        def make_actor(dev):
            kw = {"layer_norm": ln}
            if self.td3:
                kw["exploration_noise"] = hps.actor_noise_std
            cls = Actor if self.td3 else TanhGaussActor
            lo, hi = (self.min_ac.to(dev), self.max_ac.to(dev)) if dev != "meta" else (self.min_ac, self.max_ac)
            return cls(ob_shape, ac_shape, HID_DIMS, lo, hi, **kw, device=dev)

        init_actor = make_actor("cpu")  # reference init (orthogonal / zeros / ones), then moved into the arena
        self.actor = make_actor(self.device)
        self.actor.load_state_dict(init_actor.state_dict())
        self.actor.bind(ar.named(lay.actor, L.REGION_P), ar.named(lay.actor, L.REGION_G), copy_from_self=True)
        self.actor_params = dict(self.actor.named_parameters())
        self.actor_target = ar.named(lay.actor, L.REGION_T)
        self.actor_detach = make_actor(self.device)
        self.actor_detach.bind(ar.named(lay.actor, L.REGION_P), requires_grad=False)

        self.qnet1 = Critic(ob_shape, ac_shape, HID_DIMS, layer_norm=ln, device="cpu")
        self.qnet2 = Critic(ob_shape, ac_shape, HID_DIMS, layer_norm=ln, device="cpu")
        for k, q in enumerate((self.qnet1, self.qnet2)):
            q.bind(ar.named(lay.critic[k], L.REGION_P), ar.named(lay.critic[k], L.REGION_G), copy_from_self=True)
        self.qnet = Critic(ob_shape, ac_shape, HID_DIMS, layer_norm=ln, device="meta")
        self.qnet.bind(ar.stacked(L.REGION_P), ar.stacked(L.REGION_G))
        self.qnet_params = dict(self.qnet.named_parameters())  # [2, ...] views (agent.py:106)
        self.qnet_target = ar.stacked(L.REGION_T)
        with torch.no_grad():
            ar.region(L.REGION_T).copy_(ar.region(L.REGION_P))  # targets start as clones (agent.py:64,107)
        ar.sync_shadows()

        # ---- optimizers (state in arena regions 2/3)
        self.q_optimizer = ArenaAdam(self, self.qnet_params, ar.stacked(L.REGION_M), ar.stacked(L.REGION_V),
                                     hps.qnets_lr, L.CTR_Q, [(lay.critic[0].begin, lay.critic[1].end)])
        self.actor_optimizer = ArenaAdam(self, self.actor_params, ar.named(lay.actor, L.REGION_M),
                                         ar.named(lay.actor, L.REGION_V), hps.actor_lr, L.CTR_PI,
                                         [(lay.actor.begin, lay.actor.end)])

        # ---- small device state
        self.counters = torch.zeros(8, dtype=torch.int64, device=self.device)
        self.out = torch.zeros(8, dtype=torch.float32, device=self.device)
        self._alpha_state = torch.zeros(8, dtype=torch.float32, device=self.device)  # {log_alpha, grad, m, v, -}
        self._sumsq = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._sumsq_scratch = torch.zeros(64, dtype=torch.float32, device=self.device)
        self._ws: dict[int, torch.Tensor] = {}
        self._staging: dict[int, torch.Tensor] = {}
        self._predict_draw = 0
        self._lo: Optional[torch.Tensor] = None  # 3xTF32 mirror of the online / target regions (wide path), see lo_mirror()
        self.autotune = False
        # agent.py:134 fixes the target entropy at -A; a config may set it (a population member exported with its own value)
        targ_ent = hp_get(hps, "targ_ent")
        targ_ent = -self.ac_dim if targ_ent is None else float(targ_ent)
        if not self.td3:
            self._alpha_state[0] = math.log(hps.alpha_init)
            self.log_alpha = self._alpha_state[0:1].view(())  # 0-dim view, agent.py:128
            self.autotune = bool(hps.autotune)
            if self.autotune:
                self.targ_ent = targ_ent
                self.alpha_optimizer = ArenaAdam(self, {"log_alpha": self.log_alpha},
                                                 {"log_alpha": self._alpha_state[2:3].view(())},
                                                 {"log_alpha": self._alpha_state[3:4].view(())},
                                                 hps.log_alpha_lr, L.CTR_ALPHA, [])

        self._hyper = L.Hyper(
            td3=int(self.td3), bcq_mix=int(bool(hps.bcq_style_targ_mix)),
            targ_smoothing=int(bool(hps.targ_actor_smoothing)) if self.td3 else 0,
            autotune=int(self.autotune), gamma=float(hps.gamma),
            td3_std=float(hps.td3_std) if self.td3 else 0.0, td3_c=float(hps.td3_c) if self.td3 else 0.0,
            targ_ent=float(targ_ent), seed=self.seed)
        self.info = [log_module_info(m) for m in (self.actor, self.qnet1, self.qnet2)]

    # ------------------------------------------------------------------ plumbing
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def workspace(self, batch: int) -> torch.Tensor:
        if batch not in self._ws:
            n = self._lib.b2rl_workspace_floats(batch)
            if n < 0:
                raise L.B2rlError(f"batch size {batch} must be >= 1")
            self._ws[batch] = torch.zeros(n, dtype=torch.float32, device=self.device)
        return self._ws[batch]

    def _rows_of(self, batch) -> torch.Tensor:
        if isinstance(batch, Batch):
            rows = batch.rows
        elif isinstance(batch, torch.Tensor):
            rows = batch
        else:  # the reference's six-key mapping (TensorDict or dict): pack it
            n = batch["observations"].shape[0]
            rows = pack_rows(batch, self.fmt, self._staging.setdefault(
                n, torch.zeros(n, self.fmt.row_stride, dtype=torch.float32, device=self.device)))
        assert rows.is_contiguous() and rows.dtype == torch.float32 and rows.shape[1] == self.fmt.row_stride
        return rows

    def _noise(self, eps, rows) -> Optional[torch.Tensor]:
        if eps is None:
            return None
        eps = eps.to(device=self.device, dtype=torch.float32).contiguous()
        assert eps.shape == (rows.shape[0], self.ac_dim)
        return eps

    def update_args(self, rows: torch.Tensor, eps=None, eps2=None, eps_out=None, eps2_out=None,
                    dbg_targ_q=None, dbg_q=None, storage=None, storage_size: int = 0, idx_out=None,
                    new_rows=None, n_new: int = 0) -> L.UpdateArgs:
        """storage (the replay buffer's row tensor [capacity, row_stride]): the critic step samples the batch itself and
        fills `rows` / `idx_out` (include/b2rl.h, b2rl_update_args_t.storage); default: `rows` holds the batch."""
        lay, B = self.layout, rows.shape[0]
        a = L.UpdateArgs()
        a.hp, a.fmt = self._hyper, self.fmt
        a.actor = lay.actor.c_struct()
        a.critic[0], a.critic[1] = lay.critic[0].c_struct(), lay.critic[1].c_struct()
        a.batch, a.n_agents, a.agent_base = B, 1, self.agent_id
        a.region_stride, a.arena_agent_stride = lay.region, self.arena.agent_stride
        a.arena, a.rows, a.rows_agent_stride = self.arena.flat.data_ptr(), rows.data_ptr(), rows.numel()
        a.min_ac, a.max_ac = self.min_ac.data_ptr(), self.max_ac.data_ptr()
        a.log_alpha = self._alpha_state.data_ptr()
        a.eps, a.eps2, a.eps_out, a.eps2_out = L.ptr(eps), L.ptr(eps2), L.ptr(eps_out), L.ptr(eps2_out)
        a.counters = self.counters.data_ptr()
        ws = self.workspace(B)
        a.workspace, a.workspace_agent_stride = ws.data_ptr(), ws.numel()
        a.out, a.dbg_targ_q, a.dbg_q = self.out.data_ptr(), L.ptr(dbg_targ_q), L.ptr(dbg_q)
        a.storage, a.storage_agent_stride, a.storage_size = L.ptr(storage), 0 if storage is None else storage.numel(), storage_size
        a.idx_out = L.ptr(idx_out)
        if new_rows is not None:  # replay write folded into the critic step (include/b2rl.h): pinned host or device rows
            a.new_rows, a.n_new, a.capacity = new_rows.data_ptr(), int(n_new), storage.shape[0]
        a._keep = (rows, eps, eps2, eps_out, eps2_out, dbg_targ_q, dbg_q, ws, storage, idx_out, new_rows)  # keep tensors alive with the struct
        return a

    def _seg(self, begin, end, lr=0.0, *, adam, polyak, counter=0, clip=False, grad_scale=1.0) -> L.Seg:
        return L.Seg(begin, end, lr, int(adam), int(polyak), counter, grad_scale, int(clip))

    def _adam_args(self, segs: list) -> L.AdamArgs:
        a = L.AdamArgs()
        for i, s in enumerate(segs):
            a.seg[i] = s
        a.n_seg, a.n_agents = len(segs), 1
        a.polyak, a.clip_norm = float(self.hps.polyak), float(self.hps.clip_norm)
        a.beta1, a.beta2, a.eps = 0.9, 0.999, 1e-8
        a.region_stride, a.arena_agent_stride = self.layout.region, self.arena.agent_stride
        a.arena, a.counters, a.grad_sumsq = self.arena.flat.data_ptr(), self.counters.data_ptr(), self._sumsq.data_ptr()
        a.lo, a.lo_agent_stride = L.ptr(self._lo), 2 * self.layout.region  # (NULL unless the wide 3xTF32 path is in use)
        set_shadow_pairs(a, self.layout)
        return a

    def lo_mirror(self) -> torch.Tensor:
        """[1][2][region]: the "lo parts" p - tf32(p) of the online and target regions, at the parameters' own offsets —
        the second operand of the 3xTF32 tensor-core products (wide.py). Created on first use; from then on every
        Adam / Polyak launch of this agent keeps it current (b2rl_adam_args_t.lo); steps that asked for the fused
        optimizer take the three-launch form from then on (fuses_opt). Host-side writes to the parameters
        (load_params, load_from_disk do it themselves; module.load_state_dict does not) need refresh_lo().
        Create the mirror before capturing any graph of this agent: a graph captured without it keeps launching with
        lo = NULL (and, if it was captured with the fused optimizer, keeps the fused form), so the mirror goes stale."""
        if self._lo is None:
            self._lo = torch.zeros(1, 2, self.layout.region, dtype=torch.float32, device=self.device)
            self.refresh_lo()
        return self._lo

    def refresh_lo(self) -> None:
        if self._lo is not None:
            L.check(self._lib.b2rl_tc_split_lo(self.arena.flat.data_ptr(), self._lo.data_ptr(), 2 * self.layout.region, None,
                                               self._stream()), "tc_split_lo")

    def _launch_adam(self, segs: list) -> None:
        a = self._adam_args(segs)
        L.check(self._lib.b2rl_adam_polyak_multi(C.byref(a), self._stream()), "adam_polyak_multi")

    # segments used by the update functions and by engine.py
    def critic_segs(self, polyak: bool) -> list:
        lay = self.layout
        return [self._seg(lay.critic[0].begin, lay.critic[1].end, float(self.hps.qnets_lr), adam=True, polyak=polyak,
                          counter=L.CTR_Q)]

    def actor_segs(self, polyak: bool) -> list:
        lay = self.layout
        return [self._seg(lay.actor.begin, lay.actor.end, float(self.hps.actor_lr), adam=True, polyak=polyak,
                          counter=L.CTR_PI, clip=self.hps.clip_norm > 0)]

    def polyak_segs(self, critics: bool = True, actor: bool = False) -> list:
        lay, segs = self.layout, []
        if critics:
            segs.append(self._seg(lay.critic[0].begin, lay.critic[1].end, adam=False, polyak=True))
        if actor:
            segs.append(self._seg(lay.actor.begin, lay.actor.end, adam=False, polyak=True))
        return segs

    # ------------------------------------------------------------------ enqueue-only steps (graph-safe)
    def fuses_opt(self, fused_opt: bool = True) -> bool:
        """Whether a step asked for the fused optimizer (b2rl_*_update_opt) gets it: not while a lo mirror exists,
        which only the stand-alone Adam / Polyak launch keeps current."""
        return bool(fused_opt) and self._lo is None

    def enqueue_critic_step(self, args: L.UpdateArgs, extra_segs: list = (), polyak: bool = False,
                            fused_opt: bool = True, before_adam=None) -> None:
        """update_qnets incl. optimizer.step(): fused kernel + weight gradients with Adam (and Polyak) applied in the
        same launch (fused_opt), or the three-launch form (fused kernel, weight gradients, Adam/Polyak). The fused form
        does not write the 3xTF32 mirror, so an agent that has one (lo_mirror()) takes the three-launch form."""
        if self.fuses_opt(fused_opt):
            opt = self._adam_args(self.critic_segs(polyak) + list(extra_segs))
            L.check(self._lib.b2rl_critic_update_opt(C.byref(args), C.byref(opt), self._stream()), "critic_update_opt")
            return
        fn = self._lib.b2rl_critic_update_td3 if self.td3 else self._lib.b2rl_critic_update_sac
        L.check(fn(C.byref(args), self._stream()), "critic_update")
        if before_adam is not None:  # (the log block is final here: engine.py forks its publish node off this point)
            before_adam()
        self._launch_adam(self.critic_segs(polyak) + list(extra_segs))

    def enqueue_actor_step(self, args: L.UpdateArgs, polyak: bool = False, fused_opt: bool = True, before_adam=None) -> None:
        st = self._stream()
        if self.fuses_opt(fused_opt) and not self.hps.clip_norm > 0:  # (clipping needs the whole gradient's norm first)
            opt = self._adam_args(self.actor_segs(polyak))
            L.check(self._lib.b2rl_actor_update_opt(C.byref(args), C.byref(opt), st), "actor_update_opt")
            if self.autotune:
                L.check(self._lib.b2rl_alpha_update(C.byref(args), float(self.hps.log_alpha_lr), st), "alpha_update")
            return
        fn = self._lib.b2rl_actor_update_td3 if self.td3 else self._lib.b2rl_actor_update_sac
        L.check(fn(C.byref(args), st), "actor_update")
        if self.hps.clip_norm > 0:  # clip_grad_norm_ over the actor's parameters (agent.py:284-285)
            lay = self.layout
            L.check(self._lib.b2rl_grad_sumsq(self.arena.flat.data_ptr(), lay.region, self.arena.agent_stride,
                                              lay.actor.begin, lay.actor.core_end, 1, self._sumsq.data_ptr(),
                                              self._sumsq_scratch.data_ptr(), st), "grad_sumsq")
        if before_adam is not None:
            before_adam()
        self._launch_adam(self.actor_segs(polyak))
        if self.autotune:
            L.check(self._lib.b2rl_alpha_update(C.byref(args), float(self.hps.log_alpha_lr), st), "alpha_update")

    # ------------------------------------------------------------------ reference API
    @property
    def alpha(self) -> Optional[torch.Tensor]:
        return None if self.td3 else self.log_alpha.exp()

    def update_qnets(self, batch, eps: Optional[torch.Tensor] = None, **dbg) -> dict[str, torch.Tensor]:
        """agents/agent.py:183-242. ``eps`` injects the N(0,1) noise (SAC next-action sample / TD3
        smoothing); default: Philox on the device."""
        rows = self._rows_of(batch)
        self.enqueue_critic_step(self.update_args(rows, eps=self._noise(eps, rows), **dbg), fused_opt=False)
        return {"loss/qf_loss": self.out[L.OUT_QF_LOSS].clone()}

    def update_actor(self, batch, eps: Optional[torch.Tensor] = None, eps_alpha: Optional[torch.Tensor] = None,
                     **dbg) -> dict[str, torch.Tensor]:
        """agents/agent.py:244-318 (policy step, then the temperature step when autotune)."""
        rows = self._rows_of(batch)
        self.enqueue_actor_step(self.update_args(rows, eps=self._noise(eps, rows), eps2=self._noise(eps_alpha, rows),
                                                 **dbg), fused_opt=False)
        out = {"loss/actor_loss": self.out[L.OUT_ACTOR_LOSS].clone()}
        if self.td3:
            return out
        if self.autotune:
            out["loss/alpha_loss"] = self.out[L.OUT_ALPHA_LOSS].clone()
        out["vitals/alpha"] = self.alpha.detach()
        return out

    def update_targ_nets(self) -> None:
        """agents/agent.py:320-331."""
        if self.td3 or (self.qnet_updates_so_far % self.hps.crit_targ_update_freq == 0):
            self._launch_adam(self.polyak_segs(critics=True, actor=self.td3))

    def predict(self, in_td: Mapping[str, torch.Tensor], *, explore: bool,
                eps: Optional[torch.Tensor] = None) -> np.ndarray:
        """agents/agent.py:172-181: SAC mode / sample, TD3 action (+ exploration noise)."""
        return self.predict_device(in_td["observations"], explore=explore, eps=eps).cpu().numpy()

    def predict_device(self, obs: torch.Tensor, *, explore: bool, eps: Optional[torch.Tensor] = None,
                       draw: Optional[int] = None) -> torch.Tensor:
        obs = obs.to(device=self.device, dtype=torch.float32).contiguous()
        n = obs.shape[0]
        act = torch.empty(n, self.ac_dim, dtype=torch.float32, device=self.device)
        args = L.UpdateArgs()
        args.hp, args.fmt, args.actor = self._hyper, self.fmt, self.layout.actor.c_struct()
        args.arena, args.region_stride = self.arena.flat.data_ptr(), self.layout.region
        args.agent_base = self.agent_id  # part of the Philox key of the exploration noise
        args.min_ac, args.max_ac = self.min_ac.data_ptr(), self.max_ac.data_ptr()
        if eps is not None:
            eps = eps.to(device=self.device, dtype=torch.float32).contiguous()
        args.eps = L.ptr(eps)
        if draw is None:
            self._predict_draw += 1
            draw = self._predict_draw
        std = float(self.hps.actor_noise_std) if self.td3 else 0.0
        L.check(self._lib.b2rl_actor_predict(C.byref(args), obs.data_ptr(), n, int(explore), std,
                                             C.c_uint64(draw), act.data_ptr(), self._stream()),
                "actor_predict")
        return act

    def policy(self, td):
        key = "action" if self.td3 else "mode"
        td[key] = self.predict_device(td["observations"], explore=False)
        return td

    def policy_explore(self, td):
        key = "action" if self.td3 else "sample"
        td[key] = self.predict_device(td["observations"], explore=True)
        return td

    # ------------------------------------------------------------------ torch-side mirrors of the reference helpers
    def batched_qf(self, params: Mapping[str, torch.Tensor], ob, action, next_q_value=None):
        """agents/agent.py:146-157 in torch (inspection / tests; the update uses critic.cu)."""
        from torch.func import functional_call
        q = Critic((self.ob_dim,), (self.ac_dim,), HID_DIMS, layer_norm=bool(self.hps.layer_norm), device="meta")
        vals = functional_call(q, dict(params), (ob, action))
        if next_q_value is not None:
            return torch.nn.functional.mse_loss(vals.view(-1), next_q_value)
        return vals

    def pi(self, params: Mapping[str, torch.Tensor], ob):
        """agents/agent.py:159-163 in torch."""
        from torch.func import functional_call
        p = dict(params)
        p.update({k: v for k, v in self.actor.named_buffers()})
        return functional_call(self.actor, p, (ob,))

    # ------------------------------------------------------------------ checkpoints (agents/agent.py:333-371)
    def save(self, path: Path, sfx: Optional[str] = None):
        """Same dict layout as the reference. Deviation (documented in DESIGN.md): ``qnet1``/``qnet2``
        hold the LIVE critics (the reference saves their stale initial weights, SURVEY.md App. C.10) and
        ``log_alpha`` / targets are included so that training can resume."""
        path = checkpoint_path(path, sfx, self.timesteps_so_far)
        ckpt = checkpoint_dict(self.hps, self.timesteps_so_far, self.actor, self.qnet1, self.qnet2, self.actor_optimizer,
                               self.q_optimizer, self.actor_target, self.qnet_target,
                               log_alpha=None if self.td3 else self.log_alpha,
                               alpha_optimizer=self.alpha_optimizer if self.autotune else None)
        torch.save(ckpt, path)
        return path

    @torch.no_grad()
    def load_from_disk(self, path: Path):
        ckpt = torch.load(path, weights_only=False, map_location=self.device)
        self.timesteps_so_far = ckpt.get("timesteps_so_far", self.timesteps_so_far)
        self.actor.load_state_dict(ckpt["actor"])
        self.qnet1.load_state_dict(ckpt["qnet1"])
        self.qnet2.load_state_dict(ckpt["qnet2"])
        self.actor_optimizer.load_state_dict(ckpt["actor_optimizer"])
        self.q_optimizer.load_state_dict(ckpt["q_optimizer"])
        for k, v in ckpt.get("actor_target", {}).items():
            self.actor_target[k].copy_(v)
        for k, v in ckpt.get("qnet_target", {}).items():
            self.qnet_target[k].copy_(v)
        if not self.td3 and "log_alpha" in ckpt:
            self.log_alpha.copy_(ckpt["log_alpha"])
            if self.autotune and "alpha_optimizer" in ckpt:
                self.alpha_optimizer.load_state_dict(ckpt["alpha_optimizer"])
        self.arena.sync_shadows()
        self.refresh_lo()

    def load(self, wandb_run_path: str, model_name: str = "ckpt_best.pth"):
        """agents/agent.py:403-425 downloads the file from wandb; network I/O is out of scope here —
        fetch the file yourself and call ``load_from_disk``."""
        raise NotImplementedError("download the checkpoint and call Agent.load_from_disk(path)")

    # ------------------------------------------------------------------ test helpers
    @torch.no_grad()
    def load_params(self, actor: Mapping[str, torch.Tensor], q1: Mapping[str, torch.Tensor],
                    q2: Mapping[str, torch.Tensor], sync_targets: bool = True) -> None:
        """Overwrite the online nets (reference-named tensors) and re-derive targets and shadows."""
        ar, lay = self.arena, self.layout
        for net, src in ((lay.actor, actor), (lay.critic[0], q1), (lay.critic[1], q2)):
            for name, view in ar.named(net, L.REGION_P).items():
                view.copy_(src[name].to(self.device))
        if sync_targets:
            ar.region(L.REGION_T).copy_(ar.region(L.REGION_P))
        ar.sync_shadows()
        self.refresh_lo()
