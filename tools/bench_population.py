#!/usr/bin/env python
"""Throughput of a stacked population (BASELINE.json config 4) on one GPU: agent-updates/s for N agents.
    python tools/bench_population.py [--wide 3xtf32|tf32|row] [--algo sac|td3] [--sweep] [--windows W] [--rb-rows R]
                                     [--checkpoint DIR] N [N ...]
--sweep: every agent has its own learning rates, discount, Polyak rate, temperature settings and (TD3) noise, read from the
per-agent table (Population(agent_hps=...)); without it every agent uses the defaults (the table is uniform).
--checkpoint DIR: after the timed windows, the file size and wall time of Population.save and Population.load (back into the
same population) with and without the replay; the files go to DIR and are deleted after each measurement. The load follows
the save at once, so it reads the file from the page cache rather than from the disk."""
import argparse
import shutil
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from oracle import make_synthetic_transitions  # noqa: E402  (synthetic data only)
from sac_td3_cudagraphs_pytorch_b200 import sac_hps, td3_hps  # noqa: E402
from sac_td3_cudagraphs_pytorch_b200.population import Population  # noqa: E402


def sweep(n, algo, seed=0):
    """Per-agent values spread around the defaults (log-uniform rates, a range of horizons and Polyak rates)."""
    r = np.random.default_rng(seed)
    d = {"qnets_lr": 10 ** r.uniform(-4, -2.5, n), "actor_lr": 10 ** r.uniform(-4.5, -3, n), "gamma": r.uniform(0.95, 0.999, n),
         "polyak": r.uniform(0.002, 0.02, n)}
    if algo == "sac":
        d.update(log_alpha_lr=10 ** r.uniform(-4, -2.5, n), alpha_init=r.uniform(0.05, 1.0, n), targ_ent=r.uniform(-4.0, -1.0, n))
    else:
        d.update(td3_std=r.uniform(0.1, 0.3, n), td3_c=r.uniform(0.3, 0.6, n), actor_noise_std=r.uniform(0.05, 0.2, n))
    return {k: [float(x) for x in v] for k, v in d.items()}


def checkpoint_timing(pop, where):
    for replay in (True, False):
        path = Path(where) / f"population_{'replay' if replay else 'no_replay'}.ckpt"
        t0 = time.perf_counter()
        pop.save(path, replay=replay)
        t_save = time.perf_counter() - t0
        size = path.stat().st_size
        t0 = time.perf_counter()
        pop.load(path)
        torch.cuda.synchronize()
        t_load = time.perf_counter() - t0
        path.unlink()
        print(f"checkpoint N={pop.N} replay={'yes' if replay else 'no ':3s} (size {pop.size}, capacity {pop.capacity}): "
              f"{size / 1e9:7.2f} GB  save {t_save:7.2f} s ({size / 1e9 / t_save:5.2f} GB/s)  load {t_load:7.2f} s "
              f"({size / 1e9 / t_load:5.2f} GB/s)", flush=True)


def run(n, wide, algo, rb_rows=20_000, iters=None, swept=False, windows=1, ckpt_dir=None):
    td = make_synthetic_transitions(rb_rows, 11, 3, [-1.0] * 3, [1.0] * 3)
    t0 = time.time()
    hps = sac_hps() if algo == "sac" else td3_hps()
    pop = Population(range(n), 11, 3, [-1.0] * 3, [1.0] * 3, hps, "cuda", seed=1, rb_capacity=rb_rows,
                     wide=None if wide == "row" else wide, agent_hps=sweep(n, algo) if swept else None)
    pop.fill_replay(td)
    t_init = time.time() - t0
    for i in range(6):
        pop.iteration()
    torch.cuda.synchronize()
    K = iters or (30 if n >= 256 else 150)
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            pop.iteration()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        print(f"N={n:5d} {algo} {wide:7s}{' sweep' if swept else ''} {ms:9.3f} ms/iteration  {n / ms * 1e3:10.0f} agent-updates/s  "
              f"(init {t_init:.1f}s, mem {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB, finite={bool(torch.isfinite(pop.out).all())})",
              flush=True)
    if ckpt_dir:
        print(f"checkpoint dir {ckpt_dir}: {shutil.disk_usage(ckpt_dir).free / 1e9:.0f} GB free", flush=True)
        checkpoint_timing(pop, ckpt_dir)
    del pop
    torch.cuda.empty_cache()
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--wide", default="3xtf32")
    ap.add_argument("--algo", default="sac")
    ap.add_argument("--iters", type=int, default=0)
    ap.add_argument("--sweep", action="store_true", help="per-agent hyperparameters that differ between the agents")
    ap.add_argument("--windows", type=int, default=1, help="timed windows of --iters iterations each")
    ap.add_argument("--rb-rows", type=int, default=20_000, help="replay capacity, filled with as many transitions per agent")
    ap.add_argument("--checkpoint", metavar="DIR", help="also time save / load of the population (files written to DIR)")
    ap.add_argument("n", type=int, nargs="*", default=[1, 8, 64])
    a = ap.parse_args()
    for n in a.n:
        run(n, a.wide, a.algo, rb_rows=a.rb_rows, iters=a.iters or None, swept=a.sweep, windows=a.windows, ckpt_dir=a.checkpoint)


if __name__ == "__main__":
    main()
