#!/usr/bin/env python3
"""Quick device-time probe of the step kernel (development tool, not the bench contract)."""
import argparse
import ctypes
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lbm_b200 as L
from tools.make_inputs import channel_mask

ap = argparse.ArgumentParser()
ap.add_argument("--nx", type=int, default=16384)
ap.add_argument("--ny", type=int, default=16384)
ap.add_argument("--steps", type=int, default=20)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--kernel", default="auto")
ap.add_argument("--gpus", type=int, default=1)
ap.add_argument("--f64", action="store_true")
ap.add_argument("--sync-flags", action="store_true", help="in-process multi-GPU ordered by device flags")
a = ap.parse_args()
flags = {"auto": 0, "scalar": L.KERNEL_SCALAR, "vec4": L.KERNEL_VEC4, "tma": L.KERNEL_TMA, "persistent": L.KERNEL_PERSISTENT, "cluster": L.KERNEL_CLUSTER,
         "tb2": L.KERNEL_TB2, "tb3": L.KERNEL_TB3, "pairs": L.KERNEL_PAIRS}[a.kernel]
if a.sync_flags:
    flags |= L.SYNC_FLAGS
t0 = time.time()
mask = channel_mask(a.nx, a.ny)
bits = L.pack_obstacle_bits(mask)
t1 = time.time()
lat = L.Lattice(a.nx, a.ny, 0.1, 0.005, 1.85, obstacles=bits, bits=True, flags=flags, n_gpus=a.gpus, f64=a.f64)
t2 = time.time()
print("mask %.2fs create %.2fs free_cells %d" % (t1 - t0, t2 - t1, lat.info().free_cells), flush=True)
# K10's staging-wait counters, in -DLBM_EXPERIMENTS builds (tools/build_variants.py tb3_wait) only
exp_cycles = getattr(L.load_library(), "lbm_gpu_exp_tb3_cycles", None)
cyc = (ctypes.c_ulonglong * 2)()
# ... and K10's block times: busy fraction = sum of block times / (resident blocks x span of the run)
exp_blocks = getattr(L.load_library(), "lbm_gpu_exp_tb3_blocks", None)
blk = (ctypes.c_ulonglong * 4)()
lat.run_timed(3)
if exp_cycles:
    exp_cycles(cyc)
    exp_blocks(blk)
for r in range(a.reps):
    ms = lat.run_timed(a.steps)
    mlups = a.nx * a.ny * a.steps / ms / 1e3
    wait = ""
    if exp_cycles and exp_cycles(cyc) == 0 and cyc[1]:
        wait = "  K10 staging wait %.2f %% of its cycles" % (100.0 * cyc[0] / cyc[1])
    if exp_blocks and exp_blocks(blk) == 0 and blk[2]:
        span = blk[1] - blk[0]
        wait += "  K10 busy %.2f %% of %d slots over %.3f ms" % (100.0 * blk[2] / (blk[3] * span), blk[3], span * 1e-6)
    print("kernel=%s %dx%d gpus=%d steps=%d: %.3f ms/step  %.0f MLUPS  %.0f GB/s (x72B; x144B if f64)%s" %
          (a.kernel, a.nx, a.ny, a.gpus, a.steps, ms / a.steps, mlups, mlups * 72e-3, wait), flush=True)
av = lat.run(5)
print("av_vels", av)
