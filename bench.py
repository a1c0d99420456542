#!/usr/bin/env python
"""bench.py — gradient updates/sec of the SAC/TD3 learner iteration (batch 256, MuJoCo shapes).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b2rl|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is ONE learner iteration in the reference's cadence (orchestrator.py:337-352): replay sample
-> update_qnets -> (every 3rd iteration) 2 x update_actor on the same batch -> update_targ_nets.
`value` = iterations/s = gradient (critic) updates/s, summed over ranks (one independent learner per GPU,
no cross-GPU traffic: "weak" scaling). Default workload: BASELINE.json configs[1], TD3 Hopper shapes.

  --impl b2rl       this repo: CUDA graphs of hand-written sm_100a kernels (libb2rl.so)
  --impl reference  the reference's own update path on the HOST CPU cores (torch ops; the pure-torch
                    restatement in oracle/, which reproduces the reference's agents/agent.py bit for bit —
                    the reference itself needs tensordict/torchrl/omegaconf, absent from this image)
                    [--ref-device cuda: the same torch path captured in CUDA graphs, i.e. what
                    orchestrator.py:308-315 does — an extra, not the contract's reference arm]
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

WORKLOADS = {
    # name: (algo, ob_dim, ac_dim, action bound, replay rows)  — replay sized > L2 (126 MB) so that sampled
    # rows come from HBM; Hopper rows are 112 B => 2M rows = 224 MB; Humanoid rows 3088 B => 1M rows = 3.1 GB
    "td3_hopper": ("td3", 11, 3, 1.0, 2_000_000),
    "sac_hopper": ("sac", 11, 3, 1.0, 2_000_000),
    "sac_humanoid": ("sac", 376, 17, 0.4, 1_000_000),
}
HID = 256
CADENCE = "sample + critic update + 2 actor updates every 3rd iteration + polyak"


def flops_per_iteration(algo, O, A, B=256, delay=2):
    """GEMM flops of one iteration in the reference cadence (SURVEY.md §8(d) table) and of one launch of
    the dominant kernel (critic_fused): 2*B*(La + 4*Lc + 2*(H^2+H))."""
    Lc = (O + A) * HID + HID * HID + HID
    La = O * HID + HID * HID + (A if algo == "td3" else 2 * A) * HID
    critic_fused = 2 * B * (La + 4 * Lc + 2 * (HID * HID + HID))
    critic = critic_fused + 2 * B * 2 * Lc  # + weight gradients of both critics
    if algo == "sac":
        actor = 2 * B * (La + 2 * Lc + 2 * (HID * HID + HID + A * HID) + (HID * HID + 2 * A * HID) + La) \
            + 2 * B * La  # fwd, 2 critics fwd, their dX, actor dX, actor wgrad; + alpha-step forward
    else:
        actor = 2 * B * (La + Lc + (HID * HID + HID + A * HID) + (HID * HID + A * HID) + La)
    return critic + actor * delay / (delay + 1), critic_fused


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown," \
        "clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window": getattr(self, "window", "timed region")}


# ------------------------------------------------------------------------------------------ b2rl arm
def build_learner(workload, device, seed):
    from oracle import make_synthetic_transitions  # synthetic data generator only (not on the measured path)
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.engine import LearnerEngine
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer, pack_rows, row_format
    algo, O, A, bound, cap = WORKLOADS[workload]
    hps = sac_hps() if algo == "sac" else td3_hps()
    rb = ReplayBuffer(cap, device, seed=seed)
    chunk = 250_000
    fmt = row_format(O, A)
    for c0 in range(0, cap, chunk):  # fill to capacity with SURVEY §8(d) synthetic transitions
        td = make_synthetic_transitions(min(chunk, cap - c0), O, A, [-bound] * A, [bound] * A, seed=1234 + c0)
        rb.extend({k: v.to(device) for k, v in td.items()})
    torch.manual_seed(0)
    ag = Agent({"ob_shape": (4, O), "ac_shape": (4, A)}, np.full(A, -bound, np.float32), np.full(A, bound, np.float32),
               torch.device(device), hps, rb=rb, seed=seed)
    eng = LearnerEngine(ag)
    return ag, rb, eng, fmt


def time_kernel(fn, iters=200, warm=20, per_graph=20):
    """Seconds per launch of `fn` (which enqueues exactly one kernel on the current stream), timed with
    CUDA events around replays of a CUDA graph holding `per_graph` back-to-back launches, so that the
    host's launch cost (several us through ctypes) is not what is measured."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            fn()
    reps = max(1, iters // per_graph)
    for _ in range(max(1, warm // per_graph)):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (reps * per_graph) * 1e-3


DUMP_LIMIT_BYTES = 64 << 20


def timed_outputs(eng) -> dict:
    """What a caller of LearnerEngine.iteration holds after its last call: the logged losses, the batch that step
    sampled, and the online and target parameters, as host arrays (float32; the batch indices as float64, which holds
    them exactly). Inputs are seeded, so two builds given the same arguments can be compared array for array."""
    ag = eng.agent
    out = {k.replace("/", "."): v for k, v in eng.logs().items()}
    batch = eng.last_batch()
    for k in ("observations", "actions", "rewards", "next_observations", "dones"):
        out[f"batch.{k}"] = batch[k].float()
    out["batch.index"] = batch["index"].double()
    groups = {"actor": ag.actor_params, "qnet": ag.qnet_params, "qnet_target": ag.qnet_target}
    if ag.td3:
        groups["actor_target"] = ag.actor_target
    else:
        out["log_alpha"] = ag.log_alpha
    for g, params in groups.items():
        out.update({f"{g}.{n}": p for n, p in params.items()})
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def write_outputs(directory, arrays: dict) -> None:
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(d / f"{name}.npy", a)


def run_b2rl(args, rank, world, device):
    import ctypes as C
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L
    algo, O, A, bound, cap = WORKLOADS[args.workload]
    ag, rb, eng, fmt = build_learner(args.workload, device, seed=1000 + rank)
    lib = L.load()
    st = lambda: torch.cuda.current_stream().cuda_stream

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also captures the graph variants), then the timed region: K graph replays
    K, W = args.steps, args.warmup
    for i in range(W):
        eng.iteration(i)
    barrier()
    launches = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(torch.cuda.current_device()) as clk:
        barrier()
        e0.record()
        for i in range(W, W + K):
            eng.iteration(i)
            launches += eng.launches(i)
        e1.record()
        barrier()
        outputs = timed_outputs(eng) if args.dump_outputs and rank == 0 else None  # before the untimed steps below
        # nvidia-smi samples every 100 ms and the K timed steps may last less than that: keep the SAME load running
        # (untimed) until the sampler has seen it a few times, so that `clocks` describes this load and not idle
        t_load, extra = time.perf_counter(), W + K
        while len(clk.rows) < 6 and time.perf_counter() - t_load < 4.0:
            for _ in range(500):
                eng.iteration(extra)
                extra += 1
            torch.cuda.synchronize()
        clk.window = "timed region, then the same load kept running %.1f s for the 100 ms sampler" % (time.perf_counter() - t_load)
    elapsed = e0.elapsed_time(e1) * 1e-3
    if world > 1:
        t = torch.tensor([elapsed], device=device, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        elapsed = float(t)
    value = world * K / elapsed
    finite = bool(torch.isfinite(ag.out).all())
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)

    # ---- end to end through the public API (LearnerEngine.step_async / wait): per step 4 new transitions written by the
    #      host into pinned memory -> read from there by the replay-write kernel (the H2D copy) -> sample -> update(s)
    #      -> log block written into pinned host memory (the D2H copy) -> the host reads the step's critic loss.
    #      Every step's inputs are copied and every step's result is read inside the timed region. "pipelined": the
    #      host reads step t - 1's losses after launching step t (two staging slots) — a trainer that logs every
    #      step, one step late; "sync": it reads step t's losses before preparing step t + 1.
    n_env = 4
    src_rows = torch.randn(n_env, fmt.row_stride)           # "what the envs just produced" (pageable host memory)
    step_no = [W + K]

    def e2e_loop(n, pipelined):
        prev, acc = None, 0.0
        for _ in range(n):
            eng.host_rows(n_env).copy_(src_rows)             # host write of this step's inputs into pinned memory
            t = eng.step_async(step_no[0], n_env)            # replay write (reads pinned) + sample + update(s) + log block out
            step_no[0] += 1
            if pipelined:
                if prev is not None:
                    acc += float(eng.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])
                prev = t
            else:
                acc += float(eng.wait(t, as_numpy=True)[L.OUT_QF_LOSS])
        if prev is not None:
            acc += float(eng.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])
        return acc

    def timed(pipelined):
        barrier()
        t0 = time.perf_counter()
        e2e_loop(K, pipelined)
        barrier()
        el = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([el], device=device, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            el = float(t)
        return world * K / el

    e2e_loop(12, True)                                       # captures the step-graph variants (both slots)
    e2e_sync = timed(False)
    e2e_pipe = timed(True)

    # the same loop with the behaviour policy inside the step graph (SURVEY 8(f)1: Agent.predict per environment step):
    # per step also 4 observations in (pinned), 4 actions out (pinned), read by the host before it launches the next step
    src_obs = torch.randn(n_env, O)

    def policy_loop(n):
        prev, acc = None, 0.0
        for _ in range(n):
            eng.host_rows(n_env).copy_(src_rows)
            eng.host_obs(n_env).copy_(src_obs)
            t = eng.step_async(step_no[0], n_env, n_obs=n_env, explore=True)
            step_no[0] += 1
            acc += float(eng.wait_actions()[0, 0])           # the environments need the actions now
            if prev is not None:
                acc += float(eng.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])
            prev = t
        return acc + float(eng.wait(prev, as_numpy=True)[L.OUT_QF_LOSS])

    policy_loop(12)
    barrier()
    t0 = time.perf_counter()
    policy_loop(K)
    barrier()
    e2e_policy = world * K / (time.perf_counter() - t0)
    e2e = {"value": e2e_pipe, "unit": "updates/s", "h2d_bytes_per_step": n_env * fmt.row_stride * 4,
           "d2h_bytes_per_step": 32, "steps": K, "mode": "one step in flight while the host prepares the next; "
           "every step's losses are read, one step late", "sync_value": e2e_sync,
           "with_policy_value": e2e_policy, "with_policy": "the same plus Agent.predict on 4 observations inside the step graph "
           "(pinned obs in, pinned actions out, actions read before the next step is launched)"}

    if rank != 0:
        return None

    # ---- roofline of the dominant kernel (critic_fused), timed live with CUDA events on its stream
    it_flops, cf_flops = flops_per_iteration(algo, O, A)
    a = eng.args_q
    t_cf = time_kernel(lambda: L.check(lib.b2rl_launch_single(C.byref(a), 0, st())))
    per_kernel = {"critic_fused_us": t_cf * 1e6}
    per_kernel["critic_wgrad_us"] = time_kernel(lambda: L.check(lib.b2rl_launch_single(C.byref(a), 1, st()))) * 1e6
    ap = eng.args_pi[0]
    per_kernel["actor_fused_us"] = time_kernel(lambda: L.check(lib.b2rl_launch_single(C.byref(ap), 2, st()))) * 1e6
    per_kernel["actor_wgrad_us"] = time_kernel(lambda: L.check(lib.b2rl_launch_single(C.byref(ap), 3, st()))) * 1e6
    per_kernel["adam_polyak_critics_us"] = time_kernel(lambda: ag._launch_adam(ag.critic_segs(True))) * 1e6
    per_kernel["gather_us"] = time_kernel(lambda: rb.sample(256)) * 1e6
    sink = torch.zeros(4, device=device)
    fl = C.c_double(0.0)
    t_probe = time_kernel(lambda: L.check(lib.b2rl_ffma_probe(sink.data_ptr(), 4096, C.byref(fl), st())), iters=20, warm=3)
    ffma_peak = fl.value / t_probe / 1e12
    tr = REPO / "profiles" / "r2_traffic.json"  # DRAM bytes per launch from the committed ncu --set full captures
    if not tr.exists():
        tr = REPO / "profiles" / "r1_traffic.json"
    traffic = None
    if tr.exists() and args.workload == "td3_hopper":
        t_ = json.loads(tr.read_text())["critic_fused_kernel"]
        traffic = t_["dram_bytes_read"] + t_["dram_bytes_write"]
    roof = {"bound": "fp32-ffma", "kernel": "critic_fused_kernel", "achieved": cf_flops / t_cf / 1e12, "peak": ffma_peak,
            "unit": "TFLOP/s", "frac": cf_flops / t_cf / 1e12 / ffma_peak, "traffic": traffic,
            "peak_source": "measured in this run by b2rl_ffma_probe (MEASURED_PEAKS.json has only HBM and bf16 tensor peaks)",
            "flops_per_launch": cf_flops, "us_per_launch": t_cf * 1e6, "whole_step_tflops": it_flops * K / elapsed / 1e12}
    # replay gather alone at a bandwidth-relevant size (HBM roofline): 65536 rows per launch
    peaks = json.loads((REPO / "MEASURED_PEAKS.json").read_text()) if (REPO / "MEASURED_PEAKS.json").exists() else {}
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    GB = min(1 << 20, cap)  # >= 117 MB read at random + 117 MB written per launch (Hopper): out of L2, launch cost < 2 %
    t_g = time_kernel(lambda: rb.sample(GB), iters=40, warm=10, per_graph=10)
    g_bytes = GB * (2 * fmt.row_stride * 4 + 8)
    tg_ = None
    if tr.exists() and args.workload != "sac_humanoid" and "gather_kernel" in json.loads(tr.read_text()):
        t_ = json.loads(tr.read_text())["gather_kernel"]
        tg_ = t_["dram_bytes_read"] + t_["dram_bytes_write"]
    roof_g = {"bound": "hbm", "kernel": "gather_kernel", "achieved": g_bytes / t_g / 1e9, "peak": hbm_peak, "unit": "GB/s",
              "frac": g_bytes / t_g / 1e9 / hbm_peak, "traffic": tg_, "rows_per_launch": GB, "us_per_launch": t_g * 1e6,
              "bytes_per_row": 2 * fmt.row_stride * 4 + 8,
              "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"}
    rb._rows.pop(GB, None)
    rb._idx.pop(GB, None)

    # the tensor-core hidden layer of the large-batch path (BASELINE.json config 5: batch 65 536) on its own: HBM-bound
    # (X in, H and x-hat out: 3 x 4 bytes per element moved, 512 flops per element)
    MT = 65536
    Xt = torch.randn(MT, 256, device=device)
    Wt = torch.randn(256, 256, device=device) / 16
    Wlo = torch.empty_like(Wt)
    vb, vg, vbe = torch.randn(256, device=device), torch.ones(256, device=device), torch.zeros(256, device=device)
    Ht, XHt, stt = torch.empty(MT, 256, device=device), torch.empty(MT, 256, device=device), torch.empty(MT, 2, device=device)
    L.check(lib.b2rl_tc_split_lo(Wt.data_ptr(), Wlo.data_ptr(), Wt.numel(), None, st()))
    roof_tc = {}
    for tag, lo in (("3xtf32", Wlo.data_ptr()), ("tf32", None)):
        t_tc = time_kernel(lambda: L.check(lib.b2rl_tc_linear(Xt.data_ptr(), 256, MT, Wt.data_ptr(), lo, vb.data_ptr(), vg.data_ptr(),
                                                              vbe.data_ptr(), 1, 1, Ht.data_ptr(), XHt.data_ptr(), stt.data_ptr(), None, st())),
                           iters=100, warm=20)
        tc_bytes = 3 * MT * 256 * 4 + 2 * 256 * 256 * 4
        roof_tc[tag] = {"us_per_launch": t_tc * 1e6, "achieved": tc_bytes / t_tc / 1e9, "frac": tc_bytes / t_tc / 1e9 / hbm_peak,
                        "tflops": 2.0 * MT * 256 * 256 / t_tc / 1e12}
    tt = None
    if tr.exists() and "tc_linear_kernel" in json.loads(tr.read_text()):
        t_ = json.loads(tr.read_text())["tc_linear_kernel"]
        tt = t_["dram_bytes_read"] + t_["dram_bytes_write"]
    roof_tc = {"bound": "hbm", "kernel": "tc_linear_kernel<fwd, 3xTF32> (tcgen05, large-batch path, M=65536: X in, H + x-hat out)",
               "achieved": roof_tc["3xtf32"]["achieved"], "peak": hbm_peak, "unit": "GB/s", "frac": roof_tc["3xtf32"]["frac"],
               "traffic": tt, "us_per_launch": roof_tc["3xtf32"]["us_per_launch"], "tf32": roof_tc["tf32"],
               "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"}
    del Xt, Ht, XHt

    return dict(value=value, elapsed=elapsed, launches=launches, clocks=clk.summary(), e2e=e2e, roofline=roof,
                roofline_gather=roof_g, roofline_tc_linear=roof_tc, per_kernel_us=per_kernel, finite=finite, rb_rows=cap,
                row_bytes=fmt.row_stride * 4)


# ------------------------------------------------------------------------------------------ reference arm
_CPU_DATA = {}


def make_cpu_reference(workload, device="cpu", n_rows=None):
    """The reference's CPU update path on the SAME configuration as the GPU arm: same shapes, batch 256, and a replay
    buffer of the same number of rows (2 M Hopper / 1 M Humanoid transitions, six [cap, d] tensors as torchrl stores them)."""
    from oracle import OracleAgent, make_synthetic_transitions, sac_defaults, td3_defaults
    algo, O, A, bound, cap = WORKLOADS[workload]
    n_rows = n_rows or cap
    hps = sac_defaults() if algo == "sac" else td3_defaults()
    hps.adam_capturable = False
    key = (O, A, n_rows, device)
    if key not in _CPU_DATA:  # (generated in chunks: one 1 M x 376 randn needs 3 GB of temporaries)
        parts = [make_synthetic_transitions(min(250_000, n_rows - c0), O, A, [-bound] * A, [bound] * A, seed=1234 + c0, device=device)
                 for c0 in range(0, n_rows, 250_000)]
        _CPU_DATA.clear()
        _CPU_DATA[key] = {k: torch.cat([p_[k] for p_ in parts]) for k in parts[0]}
    td = _CPU_DATA[key]
    ag = OracleAgent(O, A, [-bound] * A, [bound] * A, hps, device=device, seed=0)
    gen = torch.Generator(device=device).manual_seed(4321)

    def step(i):
        idx = torch.randint(0, n_rows, (256,), generator=gen, device=device)  # RandomSampler
        batch = {k: v[idx] for k, v in td.items()}                            # per-key gather
        return ag.iteration(i, batch)
    return step


def time_cpu_reference(workload, threads, budget_s, max_steps, warm=5):
    torch.set_num_threads(threads)
    step = make_cpu_reference(workload)
    for i in range(warm):
        step(i)
    n, t0 = 0, time.perf_counter()
    while n < max_steps and (time.perf_counter() - t0) < budget_s:
        for _ in range(3):  # whole cadence periods
            step(warm + n)
            n += 1
    return n / (time.perf_counter() - t0), n


def cpu_baseline(workload, budget_s=12.0):
    cores = os.cpu_count() or 1
    r1, n1 = time_cpu_reference(workload, 1, budget_s / 2, 600)
    rN, nN = (r1, n1) if cores == 1 else time_cpu_reference(workload, cores, budget_s / 2, 600)
    best, used = (r1, 1) if r1 >= rN else (rN, cores)
    return {"value": best, "unit": "updates/s", "cores": used, "kind": "port",
            "sample": f"{n1} iterations at 1 thread ({r1:.1f}/s) and {nN} at {cores} threads ({rN:.1f}/s) of the same "
                      f"workload (same replay size as the GPU arm: {WORKLOADS[workload][4]} rows) on the host CPU; oracle = "
                      f"bit-exact restatement of the reference"}


def run_reference(args, rank):
    if rank != 0:
        return
    algo, O, A, bound, cap = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    if args.ref_device == "cuda":
        return run_reference_cuda(args)
    # pick the faster of 1 thread / all threads (tiny ops often run slower oversubscribed), then time
    r1, _ = time_cpu_reference(args.workload, 1, 4.0, 60)
    rN, _ = time_cpu_reference(args.workload, cores, 4.0, 60)
    threads = 1 if r1 >= rN else cores
    torch.set_num_threads(threads)
    step = make_cpu_reference(args.workload)
    for i in range(args.warmup):
        step(i)
    K, budget = args.steps, 150.0
    n, t0 = 0, time.perf_counter()
    while n < K and (time.perf_counter() - t0) < budget:
        step(args.warmup + n)
        n += 1
    el = time.perf_counter() - t0
    v = n / el
    line = {"impl": "reference", "metric": "gradient updates/sec (batch 256, Hopper shapes)", "value": v,
            "unit": "updates/s", "n_gpus": args.gpus, "steps": n, "warmup": args.warmup, "ms_per_step": el / n * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "algo": algo, "ob_dim": O, "ac_dim": A, "batch": 256, "hidden": "2x256+LN",
                       "replay_rows": cap, "replay_bytes": cap * 4 * ((2 * O + A + 2 + 3) & ~3), "cadence": CADENCE,
                       "execution": "torch ops on the host CPU (the reference's cuda: false path)", "device": "host cpu"},
            "cpu_baseline": {"value": v, "unit": "updates/s", "cores": threads, "kind": "port",
                             "sample": f"{n} iterations (asked {K}, budget {budget:.0f}s); 1 thread {r1:.1f}/s vs "
                                       f"{cores} threads {rN:.1f}/s in calibration"},
            "e2e": {"value": v, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def time_reference_cuda(workload, steps, warmup, device="cuda"):
    """The reference's own GPU arrangement (orchestrator.py:308-315, :338, :352) on this GPU: the torch-op update of the
    oracle (bit-exact restatement of agents/agent.py) with update_qnets and update_actor each captured in a CUDA graph the
    way tensordict's CudaGraphModule does it (static input copies per call), eager torchrl-style sampling (randint +
    one gather per key) and the eager Polyak lerp — same shapes, batch 256 and replay size as the b2rl arm, TF32 off.
    This is the "beat the reference's CUDA-graph torch path on one B200" yardstick of the north star."""
    from oracle import OracleAgent, make_synthetic_transitions, sac_defaults, td3_defaults
    algo, O, A, bound, n_rows = WORKLOADS[workload]
    dev = device
    tf32_was = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    hps = sac_defaults() if algo == "sac" else td3_defaults()
    parts = [make_synthetic_transitions(min(250_000, n_rows - c0), O, A, [-bound] * A, [bound] * A, seed=1234 + c0, device=dev)
             for c0 in range(0, n_rows, 250_000)]
    td = {k: torch.cat([p_[k] for p_ in parts]) for k in parts[0]}
    del parts
    ag = OracleAgent(O, A, [-bound] * A, [bound] * A, hps, device=dev, seed=0, torch_adam=True)
    static = {k: v[:256].clone() for k, v in td.items()}
    graphs, kernels = {}, {}

    def graphed(name, fn):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                fn(static)
        torch.cuda.current_stream().wait_stream(s)
        try:  # device kernels of one eager call = the kernel nodes the graph replays
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                fn(static)
                torch.cuda.synchronize()
            kernels[name] = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
        except Exception:
            kernels[name] = None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn(static)
        graphs[name] = (g, out)

    graphed("q", ag.update_qnets)
    graphed("pi", ag.update_actor)

    def step(i):
        idx = torch.randint(0, n_rows, (256,), device=dev)
        batch = {k: v[idx] for k, v in td.items()}
        for k in static:
            static[k].copy_(batch[k])          # CudaGraphModule's update_ of its static inputs
        graphs["q"][0].replay()
        ag.qnet_updates_so_far += 1
        if i % 3 == 0:
            for _ in range(2):
                graphs["pi"][0].replay()
        ag.update_targ_nets()

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    el = e0.elapsed_time(e1) * 1e-3
    torch.backends.cuda.matmul.allow_tf32 = tf32_was
    del td, ag, graphs
    torch.cuda.empty_cache()
    return {"value": steps / el, "unit": "updates/s", "ms_per_step": el / steps * 1e3, "steps": steps,
            "kernels_per_graph": kernels, "replay_rows": n_rows, "tf32": False,
            "what": "reference arrangement: torch ops, update_qnets / update_actor each in a CUDA graph with static-input "
                    "copies, eager sampling + Polyak (orchestrator.py:308-315, :338, :352), same GPU, same config"}


def run_reference_cuda(args):
    r = time_reference_cuda(args.workload, args.steps, args.warmup)
    print(json.dumps({"impl": "reference", "variant": "torch ops in CUDA graphs on the GPU (orchestrator.py:308-315)",
                      "metric": "gradient updates/sec (batch 256, Hopper shapes)", "value": r["value"], "unit": "updates/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                      "higher_is_better": True, "dtype": "f32", "data": "synthetic", "kernels_per_graph": r["kernels_per_graph"],
                      "config": {"workload": args.workload, "device": "cuda", "tf32": False, "replay_rows": r["replay_rows"]}}))


# ------------------------------------------------------------------------------------------ configs 4 and 5 (every N)
def _max_over_ranks(x, world, device):
    if world > 1:
        t = torch.tensor([x], device=device, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t)
    return x


def run_dp_leg(rank, world, device, B=65536, rows=1_000_000, iters=30):
    """BASELINE.json configs[4]: SAC Hopper, batch 65 536 PER GPU from a 1 M-transition replay per GPU, data-parallel
    learner (dp.DataParallelLearner on the tcgen05 wide path, 3xTF32) with one NCCL gradient all-reduce per optimizer step.
    Weak scaling: transitions/s summed over ranks; time = CUDA events, max over ranks."""
    from oracle import make_synthetic_transitions
    from sac_td3_cudagraphs_pytorch_b200 import _lib as L, sac_hps
    from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
    from sac_td3_cudagraphs_pytorch_b200.dp import DataParallelLearner, GradComm
    from sac_td3_cudagraphs_pytorch_b200.replay import ReplayBuffer
    O, A = 11, 3
    hps = sac_hps(batch_size=B)
    rb = ReplayBuffer(rows, device, seed=77 + rank, agent_id=rank)
    for c0 in range(0, rows, 250_000):
        td = make_synthetic_transitions(min(250_000, rows - c0), O, A, [-1.0] * A, [1.0] * A, seed=4321 + c0 + 17 * rank)
        rb.extend({k: v.to(device) for k, v in td.items()})
    torch.manual_seed(0)  # identical initial parameters on every rank
    ag = Agent({"ob_shape": (O,), "ac_shape": (A,)}, np.full(A, -1.0, np.float32), np.full(A, 1.0, np.float32),
               torch.device(device), hps, rb=rb, seed=5, agent_id=rank)
    dp = DataParallelLearner(ag, rb, B, GradComm(), wide="3xtf32")
    for i in range(9):  # every (actor?, polyak?) variant: first occurrence eager, second captured, third replayed
        dp.iteration(i)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(9, 9 + iters):
        dp.iteration(i)
    e1.record()
    torch.cuda.synchronize()
    ms = _max_over_ranks(e0.elapsed_time(e1) / iters, world, device)
    # the gradient all-reduce alone (the critic bucket: both critics' gradient span)
    lay = ag.layout
    bucket = ag.arena.flat[0, L.REGION_G, lay.critic[0].begin:lay.critic[1].core_end]
    ar_us = None
    if world > 1:
        for _ in range(5):
            torch.distributed.all_reduce(bucket)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            torch.distributed.all_reduce(bucket)
        e1.record()
        torch.cuda.synchronize()
        ar_us = _max_over_ranks(e0.elapsed_time(e1) / 50 * 1e3, world, device)
    finite = bool(torch.isfinite(ag.out).all())
    out = {"ms_per_iteration": ms, "transitions_per_s": world * B / ms * 1e3, "batch_per_gpu": B, "replay_rows_per_gpu": rows,
           "precision": "3xtf32 (fp32-class gradients on tcgen05)", "graph_replay": bool(dp.graphs), "n_gpus": world,
           "allreduce_bucket_bytes": int(bucket.numel() * 4), "allreduce_us": ar_us, "scaling": "weak", "outputs_finite": finite,
           "what": "SAC Hopper, reference cadence (critic step + 2 actor/alpha steps every 3rd iteration + Polyak), gradients "
                   "all-reduced (NCCL, sum) once per optimizer step, 1/W folded into Adam"}
    del dp, ag, rb
    torch.cuda.empty_cache()
    return out


def run_population_leg(rank, world, device, n_total=1024, iters=30, rb_rows=20_000, weak=False):
    """BASELINE.json configs[3]: a population of independent SAC Hopper agents (own parameters, optimizer state, replay
    slice, Philox streams), stacked on the tcgen05 wide path, sharded over the ranks as a partition of the agent ids with
    NO cross-GPU traffic. weak=False: 1024 agents in total (shard(1024, W, rank)); weak=True: 1024 agents per GPU."""
    from oracle import make_synthetic_transitions
    from sac_td3_cudagraphs_pytorch_b200 import sac_hps
    from sac_td3_cudagraphs_pytorch_b200.population import Population, shard
    ids = range(rank * n_total, (rank + 1) * n_total) if weak else shard(n_total, world, rank)
    td = make_synthetic_transitions(rb_rows, 11, 3, [-1.0] * 3, [1.0] * 3, seed=99)
    pop = Population(ids, 11, 3, [-1.0] * 3, [1.0] * 3, sac_hps(), device, seed=1, rb_capacity=rb_rows, wide="3xtf32")
    pop.fill_replay(td)
    for i in range(6):
        pop.iteration()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        pop.iteration()
    e1.record()
    torch.cuda.synchronize()
    ms = _max_over_ranks(e0.elapsed_time(e1) / iters, world, device)
    peaks = json.loads((REPO / "MEASURED_PEAKS.json").read_text()) if (REPO / "MEASURED_PEAKS.json").exists() else {}
    hbm, tens = peaks.get("hbm_gbs", 6650.0), peaks.get("bf16_tflops_sustained", 1351.5)
    n_all = n_total * world if weak else n_total
    n_local = len(ids)
    # SURVEY §8(d): 8.6 GB of unavoidable optimizer / weight traffic and 515.6 GFLOP per iteration of 1024 agents
    floor_gb, gflop = 8.6 * n_local / 1024, 515.6 * n_local / 1024
    out = {"ms_per_iteration": ms, "agent_updates_per_s": n_all / ms * 1e3, "agent_updates_per_s_per_gpu": n_all / ms * 1e3 / world,
           "agents_total": n_all, "agents_this_rank": n_local, "n_gpus": world, "scaling": "weak" if weak else "strong",
           "hbm_floor_frac": floor_gb / (ms * 1e-3) / hbm, "tensor_frac_of_bf16_sustained": gflop / ms / tens,
           "hbm_floor": "8.6 GB per iteration of 1024 agents (Adam 28 B/param, Polyak 12 B/param, one read of the weights; SURVEY 8(d)) "
                        "/ time / MEASURED_PEAKS hbm_gbs", "precision": "3xtf32", "batch": 256, "replay_rows_per_agent": rb_rows,
           "outputs_finite": bool(torch.isfinite(pop.out).all()),
           "what": "SAC Hopper agents, batch 256 each, reference cadence; one CUDA graph replay advances every agent of the shard"}
    del pop
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3000)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--impl", default="b2rl", choices=["b2rl", "reference"])
    ap.add_argument("--workload", default="td3_hopper", choices=list(WORKLOADS))
    ap.add_argument("--ref-device", default="cpu", choices=["cpu", "cuda"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--also", default="sac_hopper,sac_humanoid", help="extra workloads measured after the main one (N=1)")
    ap.add_argument("--no-legs", action="store_true", help="skip the config-4 (population) and config-5 (data-parallel) legs")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the main workload's last timed step computed "
                    "(losses, sampled batch, online and target parameters) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b2rl":
        ap.error("--dump-outputs needs --impl b2rl")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    assert torch.cuda.is_available(), "bench.py --impl b2rl needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    device = f"cuda:{local}"
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=torch.device(device))
    res = run_b2rl(args, rank, world, device)
    extra = {}
    if rank == 0 and world == 1 and args.also:
        for w in [x for x in args.also.split(",") if x and x != args.workload]:
            a2 = argparse.Namespace(**vars(args))
            a2.workload, a2.dump_outputs = w, None
            r2 = run_b2rl(a2, 0, 1, device)
            extra[w] = {"updates_per_s": r2["value"], "ms_per_step": r2["elapsed"] / a2.steps * 1e3,
                        "e2e_updates_per_s": r2["e2e"]["value"], "critic_fused_frac_of_ffma_peak": r2["roofline"]["frac"],
                        "per_kernel_us": r2["per_kernel_us"], "roofline_gather": r2["roofline_gather"]}
            torch.cuda.empty_cache()
            if not args.no_torch_baseline:
                extra[w]["torch_cudagraph_baseline"] = time_reference_cuda(w, 300, 20, device)
            if not args.no_cpu_baseline:
                extra[w]["cpu_baseline"] = cpu_baseline(w, budget_s=8.0)
    legs = {}
    if not args.no_legs:  # BASELINE.json configs[3] and [4], at every N
        torch.cuda.empty_cache()
        legs["dp_b65536"] = run_dp_leg(rank, world, device)
        legs["population_1024"] = run_population_leg(rank, world, device)
        if world > 1:
            legs["population_1024_per_gpu"] = run_population_leg(rank, world, device, weak=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    algo, O, A, bound, cap = WORKLOADS[args.workload]
    line = {
        "metric": "gradient updates/sec (batch 256, Hopper shapes)", "value": res["value"], "unit": "updates/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["elapsed"] / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "algo": algo, "ob_dim": O, "ac_dim": A, "batch": 256, "hidden": "2x256+LN",
                   "replay_rows": res["rb_rows"], "replay_bytes": res["rb_rows"] * res["row_bytes"],
                   "l2": "inputs larger than L2: sampled rows come from a replay buffer > 126 MB; parameters/optimizer "
                         "state (8 MB) are reused every step by the nature of the loop",
                   "cadence": CADENCE, "execution": "one CUDA graph replay per step",
                   "parallelism": f"{world} independent learner(s), one per GPU, no collective"},
        "clocks": res["clocks"], "e2e": res["e2e"], "gpu_launches": res["launches"],
        "roofline": res["roofline"], "roofline_gather": res["roofline_gather"], "roofline_tc_linear": res["roofline_tc_linear"], "per_kernel_us": res["per_kernel_us"],
        "outputs_finite": res["finite"],
    }
    if extra or legs:
        line["also"] = {**extra, **legs}
    if world == 1 and not args.no_torch_baseline:
        line["torch_cudagraph_baseline"] = time_reference_cuda(args.workload, 300, 20, device)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(args.workload)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
