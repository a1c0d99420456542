"""A population of independent SAC/TD3 learners stacked on one GPU (BASELINE.json config 4).

The reference's only scale-out story is one OS process per (env, seed) (spawner.py:148-178). Here N
learners — each with its own parameters, optimizer state, replay slice, step counters and Philox streams —
live in one arena `[N, 5, region]` and every kernel of the update takes the agent index from
`blockIdx.y`, so one graph replay advances all N learners by one iteration of orchestrator.py:337-352.
Nothing is shared and nothing is reduced between agents; sharding a population over GPUs is a partition
of the agent ids (`shard`) with no collective, and because every random draw is keyed on the GLOBAL agent
id the results do not depend on the partition (tests/test_gpu_population.py).

Training against environments (the reference loop, orchestrator.py:317-352: predict -> env step -> rb.extend -> update)
runs N seeds at once: `predict` (the stacked behaviour policy) and `extend` (every agent appends n transitions to its own
slice) are the eager collection path before learning starts; `step_async` / `wait` / `wait_actions` run policy, replay
write, iteration and the log block as ONE graph replay per step, like LearnerEngine.step_async for one learner
(tests/test_gpu_population_step.py).

Members may differ in their hyperparameters (a sweep, `agent_hps`), and these may change during training
(population-based training: `set_agent_hps`, `exploit`). The kernels read them from a per-agent table in device memory
(include/b2rl.h b2rl_agent_hp_t), so a changed value reaches the next graph replay without a recapture.

A population's learner state is saved with `save` and read back in place with `load`, also by a population that holds
a different partition of the same global ids (re-sharding); `save_agent` exports one member as an Agent checkpoint
(tests/test_gpu_population_checkpoint.py).

A population sharded over the ranks of a process group is one population for PBT: `all_gather` puts every agent's score
in global id order on every rank, and `exploit_many` moves learner states between any global ids — device copies on a
rank, point-to-point transfers between ranks — with the result of a single-rank population that did the same exploits
(tests/test_gpu_population_pbt.py).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import math
import operator
import os
from pathlib import Path
from types import SimpleNamespace
from typing import Mapping, NamedTuple, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from .agents.agent import HID_DIMS, ArenaAdam, checkpoint_dict, checkpoint_path
from .hps import hp_get
from .agents.nets import Actor, Critic, TanhGaussActor
from .arena import Arena, make_layout, set_shadow_pairs
from .replay import pack_rows, row_format
from .staging import StepStaging


def shard(n_total: int, world: int, rank: int) -> range:
    """Agent ids owned by `rank`: contiguous blocks, sizes differing by at most one."""
    q, r = divmod(n_total, world)
    lo = rank * q + min(rank, r)
    return range(lo, lo + q + (1 if rank < r else 0))


# the hyperparameters that may differ between the members of one population: all of them are read by the kernels from the
# per-agent table (alpha_init only sets the initial log alpha on the host). Everything else changes launch shapes or which
# graph variant runs, and is the same for every member.
SWEEPABLE = ("qnets_lr", "actor_lr", "log_alpha_lr", "gamma", "polyak", "td3_std", "td3_c", "clip_norm", "actor_noise_std",
             "alpha_init", "targ_ent")
_ABSENT = {"log_alpha_lr": 0.0, "alpha_init": 1.0, "td3_std": 0.0, "td3_c": 0.0, "actor_noise_std": 0.0, "clip_norm": 0.0}


def _check_hp_value(key: str, v, wide: bool) -> float:
    try:
        v = float(v)
    except (TypeError, ValueError):
        raise L.B2rlError(f"agent_hps: {key} = {v!r} is not a number") from None
    if not math.isfinite(v):
        raise L.B2rlError(f"agent_hps: {key} = {v} must be finite")
    if key.endswith("_lr") and v < 0:
        raise L.B2rlError(f"agent_hps: {key} = {v} must be >= 0")
    if key == "gamma" and not 0 < v <= 1:
        raise L.B2rlError(f"agent_hps: gamma = {v} must be in (0, 1]")
    if key == "polyak" and not 0 <= v <= 1:
        raise L.B2rlError(f"agent_hps: polyak = {v} must be in [0, 1]")
    if key in ("td3_std", "td3_c", "actor_noise_std", "clip_norm") and v < 0:
        raise L.B2rlError(f"agent_hps: {key} = {v} must be >= 0")
    if key == "alpha_init" and not v > 0:
        raise L.B2rlError(f"agent_hps: alpha_init = {v} must be > 0")
    if key == "clip_norm" and v > 0 and wide:
        raise L.B2rlError(f"agent_hps: clip_norm = {v}: the tensor-core (wide) actor step has no gradient clipping")
    return v


def agent_hp_values(hps, n: int, ac_dim: int, agent_hps=None, wide: bool = False) -> list:
    """The effective sweepable values of each of n agents: `hps` (targ_ent defaults to -ac_dim), overridden by agent_hps —
    a mapping {key: n values} or a sequence of n override mappings. Raises B2rlError on a key that may not differ
    between agents (it sets launch shapes or graph variants), a wrong length or an out-of-range value."""
    base = {k: hp_get(hps, k, _ABSENT.get(k)) for k in SWEEPABLE}
    if base["targ_ent"] is None:
        base["targ_ent"] = -float(ac_dim)
    cols: dict = {}
    if agent_hps is None:
        pass
    elif isinstance(agent_hps, Mapping):
        for k, vs in agent_hps.items():
            if isinstance(vs, (str, bytes)) or not hasattr(vs, "__len__") or len(vs) != n:
                raise L.B2rlError(f"agent_hps[{k!r}]: expected a sequence of {n} values (one per agent), got {vs!r}")
            cols[k] = list(vs)
    else:
        rows = list(agent_hps)
        if len(rows) != n:
            raise L.B2rlError(f"agent_hps: expected {n} override mappings (one per agent), got {len(rows)}")
        for g, r in enumerate(rows):
            for k, v in dict(r).items():
                cols.setdefault(k, [base.get(k, hp_get(hps, k))] * n)[g] = v
    for k, vs in cols.items():
        if k not in SWEEPABLE and any(v != hp_get(hps, k) for v in vs):
            raise L.B2rlError(f"agent_hps: {k!r} cannot differ between the agents of a population (it changes launch shapes "
                              f"or graph variants); every agent uses hps.{k} = {hp_get(hps, k)!r}. Per-agent keys: "
                              f"{', '.join(SWEEPABLE)}")
    out = []
    for g in range(n):
        d = {k: _check_hp_value(k, cols[k][g] if k in cols else base[k], wide) for k in SWEEPABLE}
        out.append(d)
    return out


def agent_hp_table(values: list, td3: bool) -> np.ndarray:
    """The b2rl_agent_hp_t rows [n, 16] float32 of these effective values. An agent with clip_norm <= 0 does not clip:
    +inf there makes its clip factor min(1, inf / (norm + 1e-6)) exactly 1 when another agent's clipping launches the
    clipped optimizer step. SAC stores no TD3 noise (td3_std / td3_c / explore_std = 0), as the scalar path passes."""
    t = np.zeros((len(values), C.sizeof(L.AgentHp) // 4), dtype=np.float32)
    for g, v in enumerate(values):
        r = L.AgentHp()
        r.lr[L.CTR_Q], r.lr[L.CTR_PI], r.lr[L.CTR_ALPHA] = v["qnets_lr"], v["actor_lr"], v["log_alpha_lr"]
        r.gamma, r.polyak, r.targ_ent = v["gamma"], v["polyak"], v["targ_ent"]
        r.td3_std, r.td3_c = (v["td3_std"], v["td3_c"]) if td3 else (0.0, 0.0)
        r.explore_std = v["actor_noise_std"] if td3 else 0.0
        r.clip_norm = v["clip_norm"] if v["clip_norm"] > 0 else math.inf
        t[g] = np.frombuffer(bytes(r), dtype=np.float32)
    return t


def _graph_variant_problem(v: dict, clip: bool, autotune: bool, alpha_steps: bool) -> Optional[str]:
    """Why per-agent values v need a graph variant that graphs captured with these flags do not contain (None: they fit)."""
    if v["clip_norm"] > 0 and not clip:
        return "clip_norm > 0 needs the clipped actor step, which this population's graphs do not contain (no agent " \
               "clipped at construction)"
    if autotune and (v["log_alpha_lr"] > 0) != alpha_steps:
        return "log_alpha_lr cannot move between 0 (gradient only) and positive rates"
    return None


# ---------------------------------------------------------------------- population-based training over a sharded population
def _normalize_pairs(pairs) -> list:
    """[(dst, src)] as Python ints; B2rlError on anything that is not a sequence of integer pairs."""
    try:
        out = [(operator.index(d), operator.index(s)) for d, s in pairs]
    except (TypeError, ValueError) as e:
        raise L.B2rlError(f"exploit_many: pairs must be a sequence of (dst, src) integer global ids ({e})") from None
    return out


def check_pairs(pairs, n_total: int) -> list:
    """The (dst, src) global ids of one PBT round, validated: every id in [0, n_total), no dst twice, no dst == src."""
    pairs = _normalize_pairs(pairs)
    seen = set()
    for d, s in pairs:
        for what, x in (("dst", d), ("src", s)):
            if not 0 <= x < n_total:
                raise L.B2rlError(f"exploit_many: {what} id {x} is outside [0, n_total = {n_total})")
        if d == s:
            raise L.B2rlError(f"exploit_many: pair ({d}, {s}): dst and src are the same agent")
        if d in seen:
            raise L.B2rlError(f"exploit_many: dst {d} appears in more than one pair")
        seen.add(d)
    return pairs


class ExploitPlan(NamedTuple):
    """What one rank does in a PBT round (global ids). copies: (dst, src) with both on this rank. snapshots: this rank's
    srcs that are also dsts — cloned before anything is written, and read from the clone. sends / recvs: (peer, dst, src)
    with src / dst on this rank and the other on peer, in ascending dst order — so rank r's sends to rank s, in order,
    are rank s's receives from r."""
    copies: list
    snapshots: list
    sends: list
    recvs: list


def plan_exploit(pairs, owner: Sequence[int], rank: int) -> ExploitPlan:
    """The plan of `rank` for validated pairs (check_pairs); owner[id] is the rank that holds global id `id`. Every dst
    ends with its src's state as it was before the round (chains and swaps included), whatever the order of the pairs."""
    pairs = sorted(pairs)
    dsts = {d for d, _ in pairs}
    copies, sends, recvs, read = [], [], [], set()
    for d, s in pairs:
        rd, rs = owner[d], owner[s]
        if rs == rank:
            read.add(s)
            (copies.append((d, s)) if rd == rank else sends.append((rd, d, s)))
        elif rd == rank:
            recvs.append((rs, d, s))
    return ExploitPlan(copies, sorted(read & dsts), sends, recvs)


class _Ranks:
    """The ranks of a process group that together hold one population: the id block, configuration and graph-variant
    flags of each, gathered once per population and group and validated (every rank reaches the same verdict)."""

    def __init__(self, pop: "Population", group):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        # gloo moves host tensors only: state travels through host buffers there (NCCL reads and writes the device rows)
        self.staged = self.world > 1 and dist.get_backend(group) == dist.Backend.GLOO
        got = self.gather((pop.base, pop.N, pop._config(), (pop._clip, pop.autotune, pop._alpha_steps)))
        for r, (_, _, cfg, _) in enumerate(got):
            for k, v in cfg.items():
                if v != got[0][2][k]:
                    raise L.B2rlError(f"sharded population: the configurations differ between ranks: {k} = {v!r} "
                                      f"on rank {r}, {got[0][2][k]!r} on rank 0")
        blocks = sorted((base, base + n, r) for r, (base, n, _, _) in enumerate(got))
        end = 0
        for lo, hi, r in blocks:
            if lo != end:
                raise L.B2rlError(f"sharded population: the ranks' id ranges {'overlap' if lo < end else 'leave a hole'}: "
                                  f"rank {r} holds [{lo}, {hi}), the ranks before it end at {end}")
            end = hi
        self.n_total = end
        self.ranges = [range(base, base + n) for base, n, _, _ in got]
        self.owner = np.empty(end, dtype=np.int64)
        for r, ids in enumerate(self.ranges):
            self.owner[ids.start:ids.stop] = r
        self.flags = [f for _, _, _, f in got]

    def gather(self, obj) -> list:
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        dist.all_gather_object(out, obj, group=self.group)
        return out

    def post(self, ops: list):
        """Post the point-to-point transfers [(send?, peer rank in the group, device tensor)] as one batch; returns the
        function that waits for them (stream-ordered on the current stream under NCCL)."""
        if not ops:
            return lambda: None
        bufs = [t.cpu() if send else torch.empty(t.shape, dtype=t.dtype) for send, _, t in ops] if self.staged else \
            [t for _, _, t in ops]
        reqs = dist.batch_isend_irecv([dist.P2POp(dist.isend if send else dist.irecv, b, group=self.group, group_peer=p)
                                       for (send, p, _), b in zip(ops, bufs)])

        def wait():
            for r in reqs:
                r.wait()
            if self.staged:
                for (send, _, t), b in zip(ops, bufs):
                    if not send:
                        t.copy_(b)
        return wait


CKPT_FORMAT, CKPT_VERSION = "b2rl-population", 1


def _copy_rows(dst: torch.Tensor, src: torch.Tensor, chunk_bytes: int = 1 << 28) -> None:
    """dst.copy_(src) between host and device in slices along dim 0: a strided side (a slice of the arena or of the replay)
    then needs at most one slice of contiguous scratch, not a copy of the whole array."""
    n = src.shape[0]
    step = max(1, chunk_bytes // max(1, src[0].numel() * src.element_size())) if n else 1
    for a in range(0, n, step):
        dst[a:a + step].copy_(src[a:a + step])


def _to_host(src: torch.Tensor) -> torch.Tensor:
    out = torch.empty(src.shape, dtype=src.dtype)
    _copy_rows(out, src)
    return out


def init_agent_params(agent_id: int, seed: int, ob_dim: int, ac_dim: int, td3: bool, layer_norm: bool,
                      min_ac: torch.Tensor, max_ac: torch.Tensor, noise_std: float = 0.1):
    """Reference initialisation (orthogonal / zeros / ones, agents/nets.py:34-49) from a CPU generator
    seeded by (seed, GLOBAL agent id): the same agent gets the same weights on any shard."""
    state, threads = torch.get_rng_state(), torch.get_num_threads()
    torch.manual_seed((int(seed) * 1_000_003 + int(agent_id)) & 0x7FFFFFFFFFFFFFFF)
    torch.set_num_threads(1)  # LAPACK's QR rounds differently with different thread counts
    try:
        kw = {"layer_norm": layer_norm}
        if td3:
            actor = Actor((ob_dim,), (ac_dim,), HID_DIMS, min_ac, max_ac, exploration_noise=noise_std, device="cpu", **kw)
        else:
            actor = TanhGaussActor((ob_dim,), (ac_dim,), HID_DIMS, min_ac, max_ac, device="cpu", **kw)
        q1 = Critic((ob_dim,), (ac_dim,), HID_DIMS, device="cpu", **kw)
        q2 = Critic((ob_dim,), (ac_dim,), HID_DIMS, device="cpu", **kw)
    finally:
        torch.set_rng_state(state)
        torch.set_num_threads(threads)
    sd = lambda m: {k: v for k, v in m.state_dict().items() if k.startswith(("fc_stack", "head"))}
    return sd(actor), sd(q1), sd(q2)


class Population:
    def __init__(self, agent_ids, ob_dim: int, ac_dim: int, min_ac, max_ac, hps, device, seed: int = 0,
                 rb_capacity: int = 100_000, batch_size: Optional[int] = None, use_graphs: bool = True,
                 wide: Optional[str] = None, agent_hps=None):
        """agent_hps: per-agent values of the SWEEPABLE keys, as {key: N values} or N override mappings (None: every agent
        uses hps). Agent g then trains exactly as a one-agent Population built with its values as plain hps.
        wide: None = the batch-256 row-group kernels with the agent in blockIdx.y (each agent's layers stream from L2
        once per 8 rows: latency-optimal for ONE agent, ~10 TFLOP/s however many are stacked); "3xtf32" / "tf32" = the
        layer-by-layer tensor-core path (wide.py) with the agents stacked along the row dimension — n_agents x batch rows
        per launch, per-agent weights fetched by rank-3 TMA maps: what a population of hundreds of agents wants."""
        self.ids = list(agent_ids)
        assert self.ids == list(range(self.ids[0], self.ids[0] + len(self.ids))), "agent ids must be contiguous"
        self.N, self.base = len(self.ids), self.ids[0]
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.B2rlError("Population needs a CUDA device (there is no CPU path)")
        self._lib = L.load()
        L.init_device(self.device)
        self.hps, self.seed = hps, int(seed)
        self.td3 = bool(hps.prefer_td3_over_sac)
        self.ob_dim, self.ac_dim = int(ob_dim), int(ac_dim)
        self.B = int(batch_size or hps.batch_size)
        self.use_graphs = use_graphs
        self.min_ac = torch.tensor(np.asarray(min_ac), dtype=torch.float, device=self.device)
        self.max_ac = torch.tensor(np.asarray(max_ac), dtype=torch.float, device=self.device)
        ln = bool(hps.layer_norm)
        self.fmt = row_format(self.ob_dim, self.ac_dim)
        self.layout = make_layout(self.ob_dim, self.ac_dim, self.td3, ln)
        self.arena = Arena(self.layout, self.device, n_agents=self.N)
        N, dev, lay = self.N, self.device, self.layout
        self.autotune = (not self.td3) and bool(hps.autotune)
        self._hp = agent_hp_values(hps, N, self.ac_dim, agent_hps, wide=bool(wide))
        # what the captured graphs fix: whether the clipped actor step runs (any agent clips) and whether the temperature
        # takes an Adam step (log_alpha_lr > 0) or leaves its gradient only (0); set_agent_hps keeps both
        self._clip = any(v["clip_norm"] > 0 for v in self._hp)
        self._alpha_steps = any(v["log_alpha_lr"] > 0 for v in self._hp)
        if self.autotune and self._alpha_steps != all(v["log_alpha_lr"] > 0 for v in self._hp):
            raise L.B2rlError("agent_hps: log_alpha_lr = 0 (temperature gradient only) cannot be mixed with positive rates")
        if self.autotune and wide and not self._alpha_steps:
            raise L.B2rlError("agent_hps: the tensor-core (wide) temperature step needs log_alpha_lr > 0")
        self.agent_hp_table = torch.from_numpy(agent_hp_table(self._hp, self.td3)).to(dev)

        for g, aid in enumerate(self.ids):
            a, q1, q2 = init_agent_params(aid, seed, ob_dim, ac_dim, self.td3, ln, self.min_ac.cpu(), self.max_ac.cpu(),
                                          self._hp[g]["actor_noise_std"] if self.td3 else 0.1)
            for net, src in ((lay.actor, a), (lay.critic[0], q1), (lay.critic[1], q2)):
                with torch.no_grad():
                    for name, view in self.arena.named(net, L.REGION_P, g).items():
                        view.copy_(src[name])
        with torch.no_grad():
            self.arena.flat[:, L.REGION_T].copy_(self.arena.flat[:, L.REGION_P])
        self.arena.sync_shadows()

        self.counters = torch.zeros(N, 8, dtype=torch.int64, device=dev)
        self.out = torch.zeros(N, 8, dtype=torch.float32, device=dev)
        self.alpha_state = torch.zeros(N, 5, dtype=torch.float32, device=dev)
        if not self.td3:
            self.alpha_state[:, 0] = torch.tensor([math.log(v["alpha_init"]) for v in self._hp], dtype=torch.float32)
        self.sumsq = torch.zeros(N, dtype=torch.float32, device=dev)
        self.sumsq_scratch = torch.zeros(N * 64, dtype=torch.float32, device=dev)
        ws = self._lib.b2rl_workspace_floats(self.B)
        if ws < 0:
            raise L.B2rlError(f"batch size {self.B} must be >= 1")
        self.workspace = torch.zeros(N, ws, dtype=torch.float32, device=dev)
        self.rows = torch.zeros(N, self.B, self.fmt.row_stride, dtype=torch.float32, device=dev)
        self.idx = torch.zeros(N, self.B, dtype=torch.int64, device=dev)
        self.capacity = int(rb_capacity)
        self.storage = torch.zeros(N, self.capacity, self.fmt.row_stride, dtype=torch.float32, device=dev)
        self.size = 0  # host mirror of every agent's replay fill count and write cursor (counters[:, SIZE / CURSOR])
        self.cursor = 0
        self.iterations = 0
        self.graphs: dict = {}
        self.launches_per_variant: dict = {}
        self._hyper = L.Hyper(
            td3=int(self.td3), bcq_mix=int(bool(hps.bcq_style_targ_mix)),
            targ_smoothing=int(bool(hps.targ_actor_smoothing)) if self.td3 else 0, autotune=int(self.autotune),
            gamma=float(hps.gamma), td3_std=float(hps.td3_std) if self.td3 else 0.0,
            td3_c=float(hps.td3_c) if self.td3 else 0.0, targ_ent=float(-self.ac_dim), seed=self.seed)
        self.args = self._make_args()  # the scalars of hps (agent_hp NULL): what a caller of the fused-optimizer entry points passes
        self._hp_args = L.UpdateArgs.from_buffer_copy(self.args)  # every launch of the population reads its table
        self._hp_args.agent_hp = self.agent_hp_table.data_ptr()
        self._lo: Optional[torch.Tensor] = None
        self.wide = wide
        self.wide_q = self.wide_pi = None
        if wide:
            from .wide import WideActor, WideCritic, _Owner
            own = _Owner(self)
            self.wide_q = WideCritic(own, self.B, wide)
            self.wide_pi = WideActor(own, self.B, wide)
        self._stage = StepStaging(dev, (N,), self.fmt.row_stride, self.ob_dim, self.ac_dim)
        self._predict_draw = 0
        self._rank_layouts: dict = {}  # process group -> _Ranks (exploit_many, all_gather, n_total)

    # ------------------------------------------------------------------ replay
    def fill_replay(self, td: Mapping[str, torch.Tensor], agent: Optional[int] = None) -> None:
        """Load transitions (the reference's six keys) into one agent's slice, or the same data into all."""
        rows = pack_rows({k: v.to(self.device) for k, v in td.items()}, self.fmt)
        n = rows.shape[0]
        assert n <= self.capacity
        if agent is None:
            self.storage[:, :n] = rows
        else:
            self.storage[agent, :n] = rows
        self.size = max(self.size, n)
        self.cursor = n % self.capacity
        self.counters[:, L.CTR_SIZE] = self.size
        self.counters[:, L.CTR_CURSOR] = self.cursor

    def _launch_extend(self, rows_ptr: int, n: int) -> None:
        L.check(self._lib.b2rl_replay_extend_dev_stack(self.storage.data_ptr(), self.storage[0].numel(), self.capacity, self.fmt,
                                                       rows_ptr, n, self.N, self.counters.data_ptr(), self._stream()),
                "replay_extend_dev_stack")

    def _advance(self, n: int) -> None:
        self.cursor = (self.cursor + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def extend(self, rows: torch.Tensor) -> None:
        """rb.extend(td) (orchestrator.py:100-113) for every agent at once: rows [N, n, row_stride] (replay.pack_rows
        layout; device or pinned host memory, which the write kernel reads itself) are appended round robin to each
        agent's slice at the shared cursor. Enqueued only: a pinned source must stay untouched until the stream has
        passed this point."""
        if not isinstance(rows, torch.Tensor) or rows.dim() != 3 or rows.shape[0] != self.N or \
                rows.shape[2] != self.fmt.row_stride or rows.dtype != torch.float32:
            raise L.B2rlError(f"extend: rows must be float32 [{self.N}, n, {self.fmt.row_stride}], got "
                              f"{getattr(rows, 'dtype', type(rows))} {tuple(getattr(rows, 'shape', ()))}")
        n = rows.shape[1]
        if not 1 <= n <= self.capacity:
            raise L.B2rlError(f"extend: n = {n} transitions per agent must be in [1, capacity = {self.capacity}]")
        rows = rows.contiguous()
        if not (rows.is_cuda or rows.is_pinned()):
            rows = rows.to(self.device)
        self._launch_extend(rows.data_ptr(), n)
        self._advance(n)

    # ------------------------------------------------------------------ behaviour policy
    def _launch_predict(self, args: L.UpdateArgs, obs_ptr: int, n: int, explore: bool, draw: int, act_ptr: int) -> None:
        std = float(self.hps.actor_noise_std) if self.td3 else 0.0
        L.check(self._lib.b2rl_actor_predict(C.byref(args), obs_ptr, n, int(explore), std, C.c_uint64(draw), act_ptr,
                                             self._stream()), "actor_predict")

    def predict(self, obs: torch.Tensor, explore: bool, eps: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Agent.predict (agents/agent.py:172-181) for every agent: obs [N, n, ob_dim] -> actions [N, n, A] (device).
        explore: SAC sample / TD3 action + exploration noise; otherwise SAC mode / TD3 action (evaluation episodes).
        The noise is Philox keyed on a host-counted draw and the global agent id (or eps [N, n, A] when given), so each
        call draws new noise and agent g's actions equal Agent(agent_id=base + g).predict_device."""
        obs = torch.as_tensor(obs).to(device=self.device, dtype=torch.float32).contiguous()
        if obs.dim() != 3 or obs.shape[0] != self.N or obs.shape[2] != self.ob_dim or obs.shape[1] < 1:
            raise L.B2rlError(f"predict: obs must be [{self.N}, n, {self.ob_dim}], got {tuple(obs.shape)}")
        n = obs.shape[1]
        act = torch.empty(self.N, n, self.ac_dim, dtype=torch.float32, device=self.device)
        args = self._hp_args
        if eps is not None:
            eps = torch.as_tensor(eps).to(device=self.device, dtype=torch.float32).contiguous()
            if tuple(eps.shape) != (self.N, n, self.ac_dim):
                raise L.B2rlError(f"predict: eps must be [{self.N}, {n}, {self.ac_dim}], got {tuple(eps.shape)}")
            args = L.UpdateArgs.from_buffer_copy(self._hp_args)
            args.eps = eps.data_ptr()
        self._predict_draw += 1
        self._launch_predict(args, obs.data_ptr(), n, explore, self._predict_draw, act.data_ptr())
        return act

    # ------------------------------------------------------------------ enqueue
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _make_args(self) -> L.UpdateArgs:
        lay = self.layout
        a = L.UpdateArgs()
        a.hp, a.fmt = self._hyper, self.fmt
        a.actor = lay.actor.c_struct()
        a.critic[0], a.critic[1] = lay.critic[0].c_struct(), lay.critic[1].c_struct()
        a.batch, a.n_agents, a.agent_base = self.B, self.N, self.base
        a.region_stride, a.arena_agent_stride = lay.region, self.arena.agent_stride
        a.arena, a.rows, a.rows_agent_stride = self.arena.flat.data_ptr(), self.rows.data_ptr(), self.rows[0].numel()
        a.min_ac, a.max_ac = self.min_ac.data_ptr(), self.max_ac.data_ptr()
        a.log_alpha = self.alpha_state.data_ptr()
        a.counters = self.counters.data_ptr()
        a.workspace, a.workspace_agent_stride = self.workspace.data_ptr(), self.workspace[0].numel()
        a.out = self.out.data_ptr()
        return a

    def _adam(self, segs) -> None:
        a = L.AdamArgs()
        for i, s in enumerate(segs):
            a.seg[i] = s
        a.n_seg, a.n_agents = len(segs), self.N
        a.polyak, a.clip_norm = float(self.hps.polyak), float(self.hps.clip_norm)  # (the table's values are used)
        a.agent_hp = self.agent_hp_table.data_ptr()
        a.beta1, a.beta2, a.eps = 0.9, 0.999, 1e-8
        a.region_stride, a.arena_agent_stride = self.layout.region, self.arena.agent_stride
        a.arena, a.counters, a.grad_sumsq = self.arena.flat.data_ptr(), self.counters.data_ptr(), self.sumsq.data_ptr()
        a.lo, a.lo_agent_stride = L.ptr(self._lo), 2 * self.layout.region
        set_shadow_pairs(a, self.layout)
        L.check(self._lib.b2rl_adam_polyak_multi(C.byref(a), self._stream()), "adam_polyak_multi")

    def lo_mirror(self) -> torch.Tensor:
        """[N][2][region] lo parts of every agent's online / target regions for the 3xTF32 products (Agent.lo_mirror);
        kept current by every Adam / Polyak launch of the population."""
        if self._lo is None:
            self._lo = torch.zeros(self.N, 2, self.layout.region, dtype=torch.float32, device=self.device)
            self.refresh_lo()
        return self._lo

    def refresh_lo(self) -> None:
        if self._lo is not None:
            stk = L.Stack(self.N, self.base, self.arena.agent_stride, 2 * self.layout.region, 0, 0, 0)
            L.check(self._lib.b2rl_tc_split_lo(self.arena.flat.data_ptr(), self._lo.data_ptr(), 2 * self.layout.region,
                                               C.byref(stk), self._stream()), "tc_split_lo")

    def _enqueue(self, do_actor: bool, do_polyak: bool) -> int:
        lib, st, lay, h = self._lib, self._stream(), self.layout, self.hps
        seg = lambda b, e, lr, adam, pol, ctr=0, clip=False: L.Seg(b, e, lr, int(adam), int(pol), ctr, 1.0, int(clip))
        n = 0
        L.check(lib.b2rl_replay_sample_gather(
            self.storage.data_ptr(), self.storage[0].numel(), 0, self.fmt, self.B, self.N, None, self.idx.data_ptr(),
            self.rows.data_ptr(), C.c_uint64(self.seed), self.counters.data_ptr(), L.CTR_Q, 0, self.base, st), "gather")
        delay = int(h.actor_update_delay) if do_actor else 0
        extra = [seg(lay.actor.begin, lay.actor.end, 0.0, False, True)] if (self.td3 and do_polyak and delay == 0) else []
        if self.wide_q is not None:  # the tensor-core path, agents stacked along the rows (launch counts: tools/bench_population.py)
            self.wide_q.update_qnets(self.rows, polyak=do_polyak, extra_segs=extra)
            for j in range(delay):
                self.wide_pi.update_actor(self.rows, polyak=self.td3 and do_polyak and j == delay - 1)
            return -1
        fn = lib.b2rl_critic_update_td3 if self.td3 else lib.b2rl_critic_update_sac
        L.check(fn(C.byref(self._hp_args), st), "critic_update")
        self._adam([seg(lay.critic[0].begin, lay.critic[1].end, float(h.qnets_lr), True, do_polyak, L.CTR_Q)] + extra)
        n += 4
        for j in range(delay):
            fn = lib.b2rl_actor_update_td3 if self.td3 else lib.b2rl_actor_update_sac
            L.check(fn(C.byref(self._hp_args), st), "actor_update")
            clip = self._clip  # any agent clips; the others have clip_norm = +inf in the table
            if clip:
                L.check(lib.b2rl_grad_sumsq(self.arena.flat.data_ptr(), lay.region, self.arena.agent_stride,
                                            lay.actor.begin, lay.actor.core_end, self.N, self.sumsq.data_ptr(),
                                            self.sumsq_scratch.data_ptr(), st), "grad_sumsq")
                n += 2
            self._adam([seg(lay.actor.begin, lay.actor.end, float(h.actor_lr), True,
                            self.td3 and do_polyak and j == delay - 1, L.CTR_PI, clip)])
            n += 3
            if self.autotune:
                L.check(lib.b2rl_alpha_update(C.byref(self._hp_args), 1.0 if self._alpha_steps else 0.0, st), "alpha_update")
                n += 1
        return n

    def _variant(self, i: int) -> tuple:
        h = self.hps
        do_actor = (i % (h.actor_update_delay + 1) == 0)
        do_polyak = self.td3 or ((self.iterations + 1) % h.crit_targ_update_freq == 0)
        return do_actor, do_polyak

    def iteration(self, i: Optional[int] = None) -> None:
        """One learner iteration (orchestrator.py:337-352) for every agent of the population."""
        i = self.iterations if i is None else i
        key = self._variant(i)
        if not self.use_graphs:
            self.launches_per_variant[key] = self._enqueue(*key)
        else:
            g = self.graphs.get(key)
            if g is None:
                g = torch.cuda.CUDAGraph()
                torch.cuda.synchronize(self.device)
                with torch.cuda.graph(g):
                    self.launches_per_variant[key] = self._enqueue(*key)
                self.graphs[key] = g
            g.replay()
        self.iterations += 1

    # ------------------------------------------------------------------ the environment-facing step
    def host_rows(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [N, n, row_stride] for the transitions of the next step (n per agent); two slots, as
        LearnerEngine.host_rows: the buffer of step t may be filled while step t - 1 runs, after wait() of step t - 2."""
        return self._stage.rows(n, slot)

    def host_obs(self, n: int, slot: Optional[int] = None) -> torch.Tensor:
        """Pinned staging buffer [N, n, ob_dim] for the observations the policy acts on in the next step; two slots."""
        return self._stage.obs(n, slot)

    def wait_actions(self) -> "np.ndarray":
        """Actions [N, n_obs, A] of the last step launched with n_obs > 0 (a view of pinned host memory; valid until the
        step two launches later). The policy runs first in the step graph: the environments can step while the
        update runs."""
        return self._stage.actions()

    def wait(self, ticket: int, as_numpy: bool = False):
        """The log block [N, 8] (_lib.OUT_* columns) of the step with this ticket, from pinned host memory; valid until
        the step two tickets later is launched."""
        return self._stage.wait(ticket, as_numpy)

    def step(self, i: Optional[int] = None, n_new: int = 0, n_obs: int = 0, explore: bool = True) -> torch.Tensor:
        """step_async + wait."""
        return self.wait(self.step_async(i, n_new, n_obs, explore))

    def step_async(self, i: Optional[int] = None, n_new: int = 0, n_obs: int = 0, explore: bool = True) -> int:
        """One step of the reference loop for every agent as ONE graph replay, without a stream synchronisation:
        the behaviour policy on the n_obs observations per agent in host_obs(n_obs) (parameters before this step's
        update; actions published to pinned memory: wait_actions()), the replay write of the n_new transitions per agent
        in host_rows(n_new), the iteration (sample over each agent's grown replay, updates, Adam / Polyak) and the log
        block (wait()). Returns a ticket; at most two steps are in flight. Needs graphs."""
        if not self.use_graphs:
            raise L.B2rlError("step_async is the graph path: build the Population with use_graphs=True")
        n_new, n_obs = int(n_new), int(n_obs)
        if not 0 <= n_new <= self.capacity or n_obs < 0:
            raise L.B2rlError(f"step_async: need 0 <= n_new <= capacity ({self.capacity}) and n_obs >= 0")
        if self.size + n_new < 1:
            raise L.B2rlError("step_async: the replay is empty (fill_replay / extend first, or pass n_new > 0)")
        slot = self._stage.begin()
        i = self.iterations if i is None else i
        key = self._variant(i) + (n_new, slot, n_obs, bool(explore))
        g = self.graphs.get(key)
        if g is None:
            g = self._capture_step(key)
        g.replay()
        if n_new:
            self._advance(n_new)
        self.iterations += 1
        return self._stage.launched(n_obs, slot)

    def _capture_step(self, key) -> torch.cuda.CUDAGraph:
        do_actor, do_polyak, n_new, slot, n_obs, explore = key
        stage = self._stage
        new_rows = stage.rows(n_new, slot) if n_new else None
        obs = stage.obs(n_obs, slot) if n_obs else None
        g = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(self.device)
        with torch.cuda.graph(g):
            n = 0
            if n_obs:  # noise keyed on each agent's critic step counter (draw = UINT64_MAX), as in LearnerEngine's step
                self._launch_predict(self._hp_args, obs.data_ptr(), n_obs, explore, 2 ** 64 - 1, stage.device_actions(n_obs).data_ptr())
                stage.publish_actions(self._lib, n_obs, slot, self._stream())
                n += 2
            if n_new:  # pinned host memory is device-addressable: the write kernel is the host->device copy
                self._launch_extend(new_rows.data_ptr(), n_new)
                n += 1
            m = self._enqueue(do_actor, do_polyak)  # (-1: the wide path does not count its launches)
            stage.publish_logs(self._lib, self.out, slot, self._stream())
        self.launches_per_variant[key] = -1 if m < 0 else n + m + 1
        self.graphs[key] = g
        return g

    # ------------------------------------------------------------------ per-agent hyperparameters, population-based training
    def agent_hps(self, g: int) -> dict:
        """The effective values of the SWEEPABLE keys of local agent g (alpha_init: its initial value)."""
        return dict(self._hp[g])

    def _agents(self, agents) -> list:
        gs = [agents] if isinstance(agents, int) else [int(g) for g in agents]
        for g in gs:
            if not 0 <= g < self.N:
                raise L.B2rlError(f"agent {g} is not a local agent index in [0, {self.N})")
        return gs

    def _check_graph_variant(self, values: list, what: str) -> None:
        """Refuse per-agent values that would need a graph variant this population's graphs do not contain."""
        for v in values:
            problem = _graph_variant_problem(v, self._clip, self.autotune, self._alpha_steps)
            if problem:
                raise L.B2rlError(f"{what}: {problem}")

    def set_agent_hps(self, agents, **values) -> None:
        """Change per-agent hyperparameters of the local agents `agents` (an index or a sequence) during training: the
        explore half of population-based training. The rows are written by a stream-ordered copy on the current stream,
        so every iteration or step launched after this call uses the new values (steps already in flight keep the old
        ones), and no graph is captured again. alpha_init is refused (use exploit or write alpha_state); so is a value
        that would need another graph: clipping when no agent clipped at construction, or moving log_alpha_lr between 0
        (gradient only) and positive."""
        gs = self._agents(agents)
        bad = [k for k in values if k not in SWEEPABLE or k == "alpha_init"]
        if bad:
            raise L.B2rlError(f"set_agent_hps: {bad[0]!r} cannot be changed per agent during training; keys: "
                              f"{', '.join(k for k in SWEEPABLE if k != 'alpha_init')}")
        new = [dict(self._hp[g], **{k: _check_hp_value(k, v, bool(self.wide)) for k, v in values.items()}) for g in gs]
        self._check_graph_variant(new, "set_agent_hps")
        rows = torch.from_numpy(agent_hp_table(new, self.td3)).pin_memory()
        for i, g in enumerate(gs):
            self.agent_hp_table[g].copy_(rows[i], non_blocking=True)
            self._hp[g] = new[i]

    def exploit(self, dst: int, src: int) -> None:
        """The exploit half of population-based training: local agent dst takes over local agent src's learner state —
        parameters, targets and Adam moments (the whole arena row, shadows included), the temperature state, the optimizer
        step counters (CTR_Q / CTR_PI / CTR_ALPHA), the 3xTF32 mirror row if there is one and the hyperparameter row — by
        stream-ordered device copies on the current stream. dst keeps its replay slice, its replay counters and its global
        id (its own random streams). Between steps only, not inside a graph capture; follow with set_agent_hps(dst, ...)
        to perturb."""
        dst, src = self._agents([dst, src])
        if dst == src:
            raise L.B2rlError("exploit: dst and src are the same agent")
        if torch.cuda.is_current_stream_capturing():
            raise L.B2rlError("exploit: not legal inside a graph capture")
        with torch.no_grad():
            self.arena.flat[dst].copy_(self.arena.flat[src])
            self.alpha_state[dst].copy_(self.alpha_state[src])
            self.counters[dst, L.CTR_Q:L.CTR_ALPHA + 1].copy_(self.counters[src, L.CTR_Q:L.CTR_ALPHA + 1])
            if self._lo is not None:
                self._lo[dst].copy_(self._lo[src])
            self.agent_hp_table[dst].copy_(self.agent_hp_table[src])
        self._hp[dst] = dict(self._hp[src])

    # ------------------------------------------------------------------ the whole population over the ranks of a process group
    def _config(self) -> dict:
        """What must be the same on every rank for learner states to move between them."""
        return {"algorithm": "td3" if self.td3 else "sac", "ob_dim": self.ob_dim, "ac_dim": self.ac_dim,
                "layer_norm": bool(self.hps.layer_norm), "wide": self.wide, "region": self.layout.region,
                "row_stride": self.fmt.row_stride}

    def _ranks(self, group) -> _Ranks:
        """The id blocks of the ranks of `group` (None: the default process group if there is one, else this rank
        alone). Collective the first time for a group: every rank of it calls."""
        key = group if group is not None else ("default" if dist.is_initialized() else None)
        r = self._rank_layouts.get(key)
        if r is None:
            r = self._rank_layouts[key] = _Ranks(self, group)
        return r

    @property
    def n_total(self) -> int:
        """The number of agents of the whole population over the ranks of the default process group (this population's
        when there is none). Collective on the first use (see exploit_many)."""
        return self._ranks(None).n_total

    def local_index(self, global_id: int) -> Optional[int]:
        """The local index of global agent id `global_id`, or None when another rank holds it."""
        g = operator.index(global_id) - self.base
        return g if 0 <= g < self.N else None

    def all_gather(self, values, group=None) -> np.ndarray:
        """Per-local-agent values [N, ...] (evaluation scores, say; a tensor or anything np.asarray takes) -> an array
        [n_total, ...] in global id order, the same on every rank of `group` (shards may differ in size). Collective."""
        ranks = self._ranks(group)
        v = values.detach().cpu().numpy() if isinstance(values, torch.Tensor) else np.asarray(values)
        got = ranks.gather(v)
        for r, a in enumerate(got):
            if a.ndim < 1 or a.shape[0] != len(ranks.ranges[r]) or a.shape[1:] != got[0].shape[1:]:
                raise L.B2rlError(f"all_gather: rank {r} passed values of shape {a.shape}; expected [{len(ranks.ranges[r])}"
                                  f"{''.join(', ' + str(x) for x in got[0].shape[1:])}] (one row per local agent)")
        out = np.empty((ranks.n_total, *got[0].shape[1:]), dtype=np.result_type(*got))
        for r, a in enumerate(got):
            out[ranks.ranges[r].start:ranks.ranges[r].stop] = a
        return out

    def _aux(self, ids: list) -> torch.Tensor:
        """The small state exploit moves for these local agents (global ids) as one float32 tensor [len(ids), 27]:
        alpha_state, the optimizer step counters CTR_Q..CTR_ALPHA (int64, bit for bit) and the hyperparameter row."""
        g = [i - self.base for i in ids]
        ctr = self.counters[g, L.CTR_Q:L.CTR_ALPHA + 1].contiguous().view(torch.float32)
        return torch.cat([self.alpha_state[g], ctr, self.agent_hp_table[g]], dim=1)

    def _set_aux(self, ids: list, aux: torch.Tensor) -> None:
        if not ids:
            return
        g = [i - self.base for i in ids]
        a, c, h = aux.split([self.alpha_state.shape[1], 2 * (L.CTR_ALPHA + 1 - L.CTR_Q), self.agent_hp_table.shape[1]], 1)
        self.alpha_state[g] = a
        # the counters' bits back as int64 through a fresh buffer: a column slice of aux cannot be viewed as int64 itself
        ctr = torch.empty(len(g), c.shape[1] // 2, dtype=torch.int64, device=aux.device)
        ctr.view(torch.float32).copy_(c)
        self.counters[g, L.CTR_Q:L.CTR_ALPHA + 1] = ctr
        self.agent_hp_table[g] = h

    def exploit_many(self, pairs, group=None) -> None:
        """One exploit round of population-based training over the whole population held by the ranks of `group` (None:
        the default process group if one is initialised, else this rank alone, with no communication). pairs: (dst, src)
        GLOBAL ids. Collective: every rank of the group calls it with the same pairs.

        The result is as if every dst took its src's learner state as it was when the call started (chains and swaps
        included), copying what exploit copies: the arena row, alpha_state, counters[CTR_Q..CTR_ALPHA], the 3xTF32 mirror
        row if this rank has one (recomputed from the arena row when the src is on another rank), the hyperparameter
        row and its host values. A dst keeps its replay slice, its replay counters, its log block and its global id.
        Pairs within a rank are device copies (a src that is also a dst is cloned first); between ranks each rank sends
        and receives only its own agents' rows, point to point (batch_isend_irecv; from and into the device tensors under
        NCCL, through host buffers under gloo). Follow with set_agent_hps on the dsts a rank holds (local_index) to
        perturb.

        Between steps only: a call inside a graph capture is refused and the current stream is synchronised first.
        Everything is validated from data gathered from every rank before any write or transfer, so every rank raises
        the same B2rlError when: an id is outside [0, n_total); a dst appears twice; dst == src; the pair lists differ
        between ranks; the populations' configurations differ between ranks (algorithm, shapes, layer_norm, wide, region,
        row stride); the ranks' id ranges overlap or leave a hole; or a src's hyperparameters need a graph variant the
        dst's population does not contain (the rules of set_agent_hps)."""
        if torch.cuda.is_current_stream_capturing():
            raise L.B2rlError("exploit_many: not legal inside a graph capture")
        ranks = self._ranks(group)
        try:
            norm, err = _normalize_pairs(pairs), None
        except L.B2rlError as e:
            norm, err = None, str(e)
        digest = None if norm is None else hashlib.sha256(repr(norm).encode()).hexdigest()
        mine = {} if norm is None else {s: self._hp[s - self.base] for _, s in norm if self.local_index(s) is not None}
        got = ranks.gather((err, digest, mine))
        for r, (e, _, _) in enumerate(got):
            if e is not None:
                raise L.B2rlError(e if ranks.world == 1 else f"{e} (on rank {r})")
        if len({dg for _, dg, _ in got}) > 1:
            raise L.B2rlError(f"exploit_many: the pair lists differ between ranks (digests {[dg[:12] for _, dg, _ in got]})")
        pairs = check_pairs(norm, ranks.n_total)
        hp = {s: v for _, _, m in got for s, v in m.items()}
        for d, s in pairs:
            r = int(ranks.owner[d])
            problem = _graph_variant_problem(hp[s], *ranks.flags[r])
            if problem:
                raise L.B2rlError(f"exploit_many: pair ({d}, {s}): agent {s}'s hyperparameters do not fit the population "
                                  f"of rank {r}: {problem}")
        plan = plan_exploit(pairs, ranks.owner, ranks.rank)
        self._between_steps("exploit_many")

        base, flat, lo = self.base, self.arena.flat, self._lo
        with torch.no_grad():
            snap = {s: (flat[s - base].clone(), None if lo is None else lo[s - base].clone()) for s in plan.snapshots}
            row = lambda s: snap[s][0] if s in snap else flat[s - base]
            lo_row = lambda s: snap[s][1] if s in snap else lo[s - base]
            copy_aux = self._aux([s for _, s in plan.copies])
            peers = lambda items: {p: [(d, s) for q, d, s in items if q == p] for p in sorted({q for q, _, _ in items})}
            sends, recvs = peers(plan.sends), peers(plan.recvs)
            ops, recv_aux = [], {}
            for p, ds in sends.items():  # per peer: the small state of every pair in one tensor, then each arena row
                ops += [(True, p, self._aux([s for _, s in ds]))] + [(True, p, row(s)) for _, s in ds]
            for p, ds in recvs.items():
                recv_aux[p] = torch.empty(len(ds), copy_aux.shape[1], dtype=torch.float32, device=self.device)
                ops += [(False, p, recv_aux[p])] + [(False, p, flat[d - base]) for d, _ in ds]
            wait = ranks.post(ops)
            for d, s in plan.copies:
                flat[d - base].copy_(row(s))
                if lo is not None:
                    lo[d - base].copy_(lo_row(s))
            self._set_aux([d for d, _ in plan.copies], copy_aux)
            wait()
            for p, ds in recvs.items():
                self._set_aux([d for d, _ in ds], recv_aux[p])
                if lo is not None:  # the mirror is the lo part of the arena row, element by element (tc_split_lo)
                    for d, _ in ds:
                        g = d - base
                        stk = L.Stack(1, d, self.arena.agent_stride, 2 * self.layout.region, 0, 0, 0)
                        L.check(self._lib.b2rl_tc_split_lo(flat[g].data_ptr(), lo[g].data_ptr(), 2 * self.layout.region,
                                                           C.byref(stk), self._stream()), "tc_split_lo")
        for d, s in pairs:
            if self.local_index(d) is not None:
                self._hp[d - base] = dict(hp[s])

    # ------------------------------------------------------------------ checkpoints
    def _between_steps(self, what: str) -> None:
        if torch.cuda.is_current_stream_capturing():
            raise L.B2rlError(f"{what}: not legal inside a graph capture")
        torch.cuda.current_stream(self.device).synchronize()

    def _hps_dict(self) -> dict:
        return dict(self.hps) if isinstance(self.hps, Mapping) else dict(vars(self.hps))

    def save(self, path, replay: bool = True) -> Path:
        """Write the learner state of this population's agents to the file `path` (one torch.save'd dict, written to
        path.tmp and then renamed, so an interrupted save never leaves a truncated file under the real name). Between
        steps only: the current stream is synchronised first (no step in flight) and a call inside a graph capture is
        refused.

        The file holds a header (format, version, hps, seed, shapes, action bounds, arena region size, row stride, replay
        capacity, wide and the GLOBAL ids of the agents) and, per agent in the order of those ids: arena regions P, T, M
        and V (not G: the backward kernels overwrite every gradient element), alpha_state, the counters, the log block,
        the rows of the hyperparameter table and their host values (agent_hps); then the host counters size, cursor,
        iterations and the predict draw, and with replay=True every agent's replay rows [:size]. The staging buffers of
        step_async are not state and are not saved. Tensors are stored on the CPU, so that a loader can torch.load the
        file with mmap=True and read only the rows it needs."""
        self._between_steps("save")
        if bool(self.counters[:, [L.CTR_TICKET, L.CTR_XTICKET]].any()):
            raise L.B2rlError("save: counters[:, CTR_TICKET / CTR_XTICKET] are not 0: a step did not complete")
        path = Path(path)
        ckpt = {
            "format": CKPT_FORMAT, "version": CKPT_VERSION, "hps": self._hps_dict(), "seed": self.seed,
            "ob_dim": self.ob_dim, "ac_dim": self.ac_dim, "min_ac": self.min_ac.tolist(), "max_ac": self.max_ac.tolist(),
            "region": self.layout.region, "row_stride": self.fmt.row_stride, "capacity": self.capacity, "wide": self.wide,
            "ids": list(self.ids),
            "arena": _to_host(self.arena.flat[:, :L.REGION_G]),
            "alpha_state": self.alpha_state.cpu(), "counters": self.counters.cpu(), "out": self.out.cpu(),
            "agent_hp_table": self.agent_hp_table.cpu(), "agent_hps": [dict(v) for v in self._hp],
            "size": self.size, "cursor": self.cursor, "iterations": self.iterations, "predict_draw": self._predict_draw,
        }
        if replay:
            ckpt["storage"] = _to_host(self.storage[:, :self.size])
        tmp = path.with_name(path.name + ".tmp")
        with open(tmp, "wb") as f:
            torch.save(ckpt, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
        return path

    def _read_checkpoint(self, p) -> dict:
        """torch.load a population checkpoint (memory-mapped) and check that its learners fit this population."""
        try:
            ck = torch.load(p, map_location="cpu", mmap=True, weights_only=False)
        except Exception as e:
            raise L.B2rlError(f"load: {p}: not a population checkpoint (format: torch.load failed: {e})") from e
        fmt = ck.get("format") if isinstance(ck, Mapping) else type(ck).__name__
        if fmt != CKPT_FORMAT:
            raise L.B2rlError(f"load: {p}: not a population checkpoint (format = {fmt!r}, expected {CKPT_FORMAT!r})")
        if ck.get("version") != CKPT_VERSION:
            raise L.B2rlError(f"load: {p}: unknown population checkpoint version = {ck.get('version')!r} "
                              f"(this code reads version {CKPT_VERSION})")
        theirs = dict(ck, prefer_td3_over_sac=bool(hp_get(ck["hps"], "prefer_td3_over_sac")),
                      layer_norm=bool(hp_get(ck["hps"], "layer_norm")))
        mine = {"prefer_td3_over_sac": self.td3, "ob_dim": self.ob_dim, "ac_dim": self.ac_dim,
                "layer_norm": bool(self.hps.layer_norm), "min_ac": self.min_ac.tolist(), "max_ac": self.max_ac.tolist(),
                "region": self.layout.region, "row_stride": self.fmt.row_stride, "seed": self.seed}
        for k, v in mine.items():
            if theirs[k] != v:
                raise L.B2rlError(f"load: {p}: {k} = {theirs[k]!r} in the file, {v!r} in this population")
        if "storage" in ck and ck["capacity"] != self.capacity:
            raise L.B2rlError(f"load: {p}: capacity = {ck['capacity']} in the file (which holds the replay), "
                              f"{self.capacity} in this population (a file saved with replay=False carries no replay)")
        return ck

    def load(self, paths) -> None:
        """Fill this population IN PLACE from the rows of one checkpoint file or a list of them (e.g. one per rank of an
        earlier run: each rank passes every rank's file, or one file of the whole population) whose global ids are
        self.ids. Every write is a copy into the existing tensors, so graphs captured before the load stay valid and the
        next iteration() / step_async() continues from the loaded state (loading an earlier checkpoint into a running
        population rewinds it). The w2n shadows come with the arena rows; a 3xTF32 mirror, if there is one, is
        recomputed. Between steps only: the current stream is synchronised first, and a call inside a graph capture is
        refused.

        Everything is validated before the first write (a refused load changes nothing); B2rlError names the key when a
        file is not a population checkpoint of a known version; the algorithm, ob_dim, ac_dim, layer_norm, min_ac / max_ac,
        region, row_stride or seed differ; capacity differs and the file holds the replay; an id of this population is in
        no file or in more than one; the files disagree on a host counter; or a loaded hyperparameter row needs a graph
        variant this population does not have (the rules of set_agent_hps).

        A file without the replay (save(replay=False)) leaves storage, the replay counters CTR_SIZE / CTR_CURSOR and the
        host size / cursor as they are: training continues bitwise only if the caller refills the same data. `wide` may
        differ between the file and this population (the state has the same layout on both paths); training continues
        bitwise only on the path that wrote the file. Everything not in the file comes from this population: batch_size,
        actor_update_delay, crit_targ_update_freq, use_graphs and the rest of its hps."""
        self._between_steps("load")
        paths = [paths] if isinstance(paths, (str, os.PathLike)) else list(paths)
        cks = [self._read_checkpoint(p) for p in paths]
        src: dict = {}  # global id -> (file, row)
        for k, ck in enumerate(cks):
            for r, aid in enumerate(ck["ids"]):
                if self.base <= aid < self.base + self.N:
                    if aid in src:
                        raise L.B2rlError(f"load: ids: agent {aid} is in more than one file ({paths[src[aid][0]]}, {paths[k]})")
                    src[aid] = (k, r)
        missing = [aid for aid in self.ids if aid not in src]
        if missing:
            raise L.B2rlError(f"load: ids: agent {missing[0]} is in none of the files {[str(p) for p in paths]}")
        used = sorted({k for k, _ in src.values()})
        for key in ("size", "cursor", "iterations", "predict_draw"):
            if len({cks[k][key] for k in used}) > 1:
                raise L.B2rlError(f"load: the files disagree on {key} ({[cks[k][key] for k in used]})")
        if len({"storage" in cks[k] for k in used}) > 1:
            raise L.B2rlError("load: storage: some of the files hold the replay and some do not")
        new_hp = [dict(cks[src[aid][0]]["agent_hps"][src[aid][1]]) for aid in self.ids]
        self._check_graph_variant(new_hp, "load")

        runs: list = []  # [file, first local agent, first row, count]
        for g, aid in enumerate(self.ids):
            k, r = src[aid]
            if runs and runs[-1][0] == k and runs[-1][2] + runs[-1][3] == r:
                runs[-1][3] += 1
            else:
                runs.append([k, g, r, 1])
        head = cks[used[0]]
        replay, size = "storage" in head, head["size"]
        cols = [c for c in range(self.counters.shape[1]) if replay or c not in (L.CTR_SIZE, L.CTR_CURSOR)]
        with torch.no_grad():
            for k, g, r, n in runs:
                ck, dst, rows = cks[k], slice(g, g + n), slice(r, r + n)
                _copy_rows(self.arena.flat[dst, :L.REGION_G], ck["arena"][rows])
                self.alpha_state[dst].copy_(ck["alpha_state"][rows])
                self.counters[dst, cols] = ck["counters"][rows][:, cols].to(self.device)
                self.out[dst].copy_(ck["out"][rows])
                self.agent_hp_table[dst].copy_(ck["agent_hp_table"][rows])
                if replay:
                    _copy_rows(self.storage[dst, :size], ck["storage"][rows])
                    self.storage[dst, size:].zero_()
        self._hp = new_hp
        if replay:
            self.size, self.cursor = size, head["cursor"]
        self.iterations, self._predict_draw = head["iterations"], head["predict_draw"]
        self.refresh_lo()

    def save_agent(self, g: int, path, sfx: Optional[str] = None, timesteps_so_far: int = 0) -> Path:
        """Export local member g as an Agent checkpoint in directory `path` (ckpt_{sfx}.pth, or .ckpt_{timesteps}ts.pth):
        Agent.save's layout (agents.agent.checkpoint_dict), which Agent.load_from_disk reads. Its hps are this
        population's with the member's effective per-agent values (agent_hps(g)) in place of the shared ones (targ_ent
        only when it is not -ac_dim), so an Agent built from ckpt["hps"] with seed = self.seed, agent_id = base + g and
        the member's replay trains as the member does. Between steps only."""
        (g,) = self._agents(g)
        self._between_steps("save_agent")
        hp = self._hp[g]
        hps = self._hps_dict()
        for k, v in hp.items():
            absent = -float(self.ac_dim) if k == "targ_ent" else _ABSENT.get(k)
            if k in hps or v != absent:
                hps[k] = v
        lay, ar, ln = self.layout, self.arena, bool(self.hps.layer_norm)
        ob, ac = (self.ob_dim,), (self.ac_dim,)
        if self.td3:
            actor = Actor(ob, ac, HID_DIMS, self.min_ac, self.max_ac, exploration_noise=0.0, layer_norm=ln, device="meta")
            actor.exploration_noise = torch.as_tensor(hp["actor_noise_std"], device=self.device)
        else:
            actor = TanhGaussActor(ob, ac, HID_DIMS, self.min_ac, self.max_ac, layer_norm=ln, device="meta")
        actor.bind(ar.named(lay.actor, L.REGION_P, g), requires_grad=False)
        q1, q2 = (Critic(ob, ac, HID_DIMS, layer_norm=ln, device="meta") for _ in range(2))
        q1.bind(ar.named(lay.critic[0], L.REGION_P, g), requires_grad=False)
        q2.bind(ar.named(lay.critic[1], L.REGION_P, g), requires_grad=False)
        own = SimpleNamespace(counters=self.counters[g])  # (ArenaAdam.state_dict reads the step from counters[counter])
        pmv = (L.REGION_P, L.REGION_M, L.REGION_V)
        actor_opt = ArenaAdam(own, *(ar.named(lay.actor, r, g) for r in pmv), hp["actor_lr"], L.CTR_PI, [])
        q_opt = ArenaAdam(own, *(ar.stacked(r, g) for r in pmv), hp["qnets_lr"], L.CTR_Q, [])
        kw = {}
        if not self.td3:
            a = self.alpha_state[g]  # {log_alpha, grad, exp_avg, exp_avg_sq, -}
            kw["log_alpha"] = a[0]
            if self.autotune:
                kw["alpha_optimizer"] = ArenaAdam(own, {"log_alpha": a[0]}, {"log_alpha": a[2]}, {"log_alpha": a[3]},
                                                  hp["log_alpha_lr"], L.CTR_ALPHA, [])
        ckpt = checkpoint_dict(hps, timesteps_so_far, actor, q1, q2, actor_opt, q_opt, ar.named(lay.actor, L.REGION_T, g),
                               ar.stacked(L.REGION_T, g), **kw)
        path = checkpoint_path(path, sfx, timesteps_so_far)
        torch.save(ckpt, path)
        return path

    # ------------------------------------------------------------------ inspection
    def agent_arena(self, g: int) -> torch.Tensor:
        return self.arena.flat[g]

    def losses(self) -> dict[str, torch.Tensor]:
        d = {"loss/qf_loss": self.out[:, L.OUT_QF_LOSS], "loss/actor_loss": self.out[:, L.OUT_ACTOR_LOSS]}
        if not self.td3:
            d["vitals/alpha"] = self.out[:, L.OUT_ALPHA]
            if self.autotune:
                d["loss/alpha_loss"] = self.out[:, L.OUT_ALPHA_LOSS]
        return d
