#!/usr/bin/env python
"""In-kernel phase timing of critic_fused (thread 0 of CTA 0, and of CTA 1 for its first pass; clock64). Needs a timing build, kept beside the product library:
   export B2RL_LIB=$PWD/sac_td3_cudagraphs_pytorch_b200/libb2rl_timing.so
   B2RL_EXTRA_NVCC_FLAGS=-DB2RL_TIMING python -m sac_td3_cudagraphs_pytorch_b200.build      # writes $B2RL_LIB
   python tools/phase_timing.py td3 | sac [O A]                                              # loads $B2RL_LIB
(profiles/r2_phase_timing_*.txt)"""
import ctypes as C, sys
from pathlib import Path
import numpy as np, torch
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from sac_td3_cudagraphs_pytorch_b200 import _lib as L, td3_hps, sac_hps
from sac_td3_cudagraphs_pytorch_b200.agents.agent import Agent
lib = L.load()
algo = sys.argv[1] if len(sys.argv) > 1 else "td3"
O, A_ = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (11, 3)  # e.g. 376 17 for Humanoid
B = 256
torch.manual_seed(0)
ag = Agent({"ob_shape": (O,), "ac_shape": (A_,)}, np.full(A_, -1.0, np.float32), np.full(A_, 1.0, np.float32),
           torch.device("cuda"), (sac_hps if algo == "sac" else td3_hps)())
rows = torch.randn(B, ag.fmt.row_stride, device="cuda"); rows[:, O + A_ + 1] = 0
a = ag.update_args(rows)
st = torch.cuda.current_stream().cuda_stream
for _ in range(5):
    L.check(lib.b2rl_launch_single(C.byref(a), 0, st))
torch.cuda.synchronize()
buf = (C.c_longlong * 64)()
lib.b2rl_debug_timing.argtypes = [C.c_void_p]
assert lib.b2rl_debug_timing(buf) == 0
t = np.array(buf[:64], dtype=np.int64)
names = { **{44 + i: f"P.warp {i} job issued" for i in range(8)}, **{52 + i: f"P.warp {i} cp.async landed" for i in range(8)}, 0: "start", 40: "P.mbar init + cluster arrive", 41: "P.warp job issued", 42: "P.cp.async landed", 43: "P.before the first trunk_fwd call", 10: "A head done", 11: "A sampled, a' sent", 21: "T head done",
         22: "twin exchange done", 23: "Q acts landed, TD target done", 34: "bwd start", 35: "bwd end"}
# first pass (trunk_fwd_full, 256 columns, no exchange): the next action A on CTA 0, the online Q on CTA 1 side by side
for base, nm in ((2, "A"), (24, "Q")):
    for o, what in ((0, "l1 products start"), (2, "l1 products+reduce end"), (3, "l1 rows end"), (5, "l2 products+reduce end"),
                    (6, "l2 rows end"), (7, "l2 stats done (inside l2 rows)")):
        names[base + o] = f"{nm}.{what}"
for o, what in enumerate(("l1 gemm start", "l1 gemm+sync end", "l1 reduce+gather+barrier end", "l1 rows end",
                          "l2 gemm+sync end", "l2 reduce+gather+barrier end", "l2 rows end")):
    names[12 + o] = f"T.{what}"
names[19] = "T.l2 stats done (inside l2 rows)"
# CTA 1's timestamps are of its own clock: counted from its own start
cta1 = {1: "start", 24: "", 26: "", 27: "", 29: "", 30: "", 33: "Q head done", 37: "a' landed"}
for k, what in cta1.items():
    names[k] = "[CTA 1] " + (what or names[k])
rel = {k: t[k] - (t[1] if k in cta1 else t[0]) for k in names}
for k in sorted((k for k in names if rel[k] >= 0 and t[k] != 0), key=lambda k: rel[k]):
    print(f"{k:2d} {names[k]:36s} total {rel[k]:7d}")
