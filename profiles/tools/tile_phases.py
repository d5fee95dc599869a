"""Per-phase cycles of the k_fused_tma step loop on bench.py's C4 (2,048 replicas x 1,000 houses, TarMAC rows, D = 10,
the in-kernel step loop over the rotating action tape): where a tile-step's time goes, and whether warp 0 (which also
runs the cluster epilogue) is later than the other warps.

Needs a library built with the phase counters (they compile to nothing otherwise):
    DRSIM_EXTRA_NVCC_FLAGS=-DDRSIM_TILE_DBG DRSIM_LIB=build_ab/tile_dbg/libdrsim.so python -m marl_demandresponse_b200._build
    DRSIM_LIB=build_ab/tile_dbg/libdrsim.so DRSIM_NO_REBUILD=1 python profiles/tools/tile_phases.py [--obs-dtype bfloat16]

Every warp accumulates clock() deltas per phase over the timed launches; the counters cost a few instructions per
phase, so the step time printed next to them is that of the debug build, not of the production kernel.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import env_prop_for  # noqa: E402
from marl_demandresponse_b200 import BatchedEnv  # noqa: E402

PHASES = ["house update", "own rows + warp sum", "barrier wait", "fold + reward", "patches + row store",
          "epilogue (thread 0)"]
WARPS, SLOTS = 8, 8

ap = argparse.ArgumentParser()
ap.add_argument("--obs-dtype", default="float32", choices=["float32", "bfloat16"])
ap.add_argument("--launches", type=int, default=40, help="timed launches of 64 steps each")
args = ap.parse_args()

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
R, N = 2048, 1000
env = BatchedEnv(env_prop_for(N), R, precision="f32", obs_layout="tarmac", noise="philox", seed=1234, obs_dtype=args.obs_dtype)
env.reset()
g = torch.Generator(device="cuda").manual_seed(1234)
tape = (torch.rand((4, R, env.sim.Ns), device="cuda", generator=g) < 0.5).to(torch.uint8)
L = env.sim._L
L.drsim_debug_tile_phases.restype = C.c_int
L.drsim_debug_tile_phases.argtypes = [C.c_void_p, C.c_int, C.c_int]
env.run(256, tape, rotate=True)
torch.cuda.synchronize()
if L.drsim_debug_tile_phases(None, 1024, 1) == 0:   # (reset only)
    sys.exit("the library has no tile phase counters: build it with DRSIM_EXTRA_NVCC_FLAGS=-DDRSIM_TILE_DBG")
steps = 64 * args.launches
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
env.run(steps, tape, rotate=True)
e1.record()
torch.cuda.synchronize()
us = 1e3 * e0.elapsed_time(e1) / steps
buf = np.zeros((1024, WARPS, SLOTS), dtype=np.uint64)
n = L.drsim_debug_tile_phases(buf.ctypes.data_as(C.c_void_p), 1024, 1)
t = buf[:n].astype(np.float64)
t = t[t[:, 0, 6] > 0]                       # CTAs that ran tiles
ts = t[:, :, 6]                             # tile-steps per CTA (the same for its 8 warps)
per = t[:, :, :6] / ts[:, :, None]          # cycles per tile-step, [cta][warp][phase]
tot = per.sum(axis=2)
print(f"C4 {R} x {N}, rows {args.obs_dtype}, {steps} steps in {args.launches} launches: {us:.2f} us/step (debug build), "
      f"{len(t)} CTAs, {ts[:, 0].mean():.0f} tile-steps per CTA")
print("cycles per tile-step, mean over CTAs")
print(f"  {'phase':32s} {'all warps':>9s} {'share':>8s} {'warp 0':>8s} {'warps 1-7':>9s}")
for k, name in enumerate(PHASES):
    a, w0, wr = per[:, :, k].mean(), per[:, 0, k].mean(), per[:, 1:, k].mean()
    print(f"  {name:32s} {a:9.0f} {100 * a / tot.mean():6.1f} % {w0:8.0f} {wr:9.0f}")
print(f"  {'total':32s} {tot.mean():9.0f} {100.0:6.1f} % {tot[:, 0].mean():8.0f} {tot[:, 1:].mean():9.0f}")
late = per[:, :, :2].sum(axis=2)             # work before the barrier
print(f"work before the barrier (house + rows): warp 0 {late[:, 0].mean():.0f}, warps 1-7 {late[:, 1:].mean():.0f} cycles; "
      f"barrier wait: warp 0 {per[:, 0, 2].mean():.0f}, warps 1-7 {per[:, 1:, 2].mean():.0f}")
