#!/usr/bin/env python3
"""Parameter-sweep throughput: B lattices in one lbm_gpu_run_batch against the same B
lattices run one after another with lbm_gpu_run (development tool, not the bench contract).

For each shipped small grid (its mask and step count) and each B, the members differ in
omega.  The batch and the sequential runs alternate, --reps times each, in one process; times
are device times (CUDA events of the library, last_run_device_ms).  After the last repetition
every member's lattice digest and av_vels are compared bit for bit with its sequential twin.
Prints one JSON line per (grid, B) after a line naming the GPU and its power limit.

  python tools/batch_bench.py [--grids 128x128,128x256,256x256] [--batches 1,2,4,...] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbm_b200 as L
from tools.make_inputs import SHIPPED, shipped_mask


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or "unknown"


def lattices(name, b):
    nx, ny, _iters, _re, rho, acc, om, _r, _c = SHIPPED[name]
    obst = shipped_mask(name).astype(np.int32)
    return [L.Lattice(nx, ny, rho, acc, om - 0.01 * i, obstacles=obst) for i in range(b)]


def measure(name, b, steps, reps, warmup):
    nx, ny = SHIPPED[name][:2]
    batch, solo = lattices(name, b), lattices(name, b)
    L.run_batch(batch, warmup)
    for lat in solo:
        lat.run(warmup)
    t_batch, t_seq = [], []
    for _ in range(reps):
        av_b = L.run_batch(batch, steps)
        t_batch.append(batch[0].info().last_run_device_ms)
        av_s, ms = [], 0.0
        for lat in solo:
            av_s.append(lat.run(steps))
            ms += lat.info().last_run_device_ms
        t_seq.append(ms)
    same = all(np.array_equal(av_b[i].view(np.uint32), av_s[i].view(np.uint32)) and
               batch[i].digest() == solo[i].digest() for i in range(b))
    for lat in batch + solo:
        lat.close()
    cells = b * nx * ny * steps
    tb, ts = float(np.median(t_batch)), float(np.median(t_seq))
    return {"grid": name, "B": b, "steps": steps, "reps": reps,
            "batch_ms": round(tb, 3), "batch_ms_spread": [round(min(t_batch), 3), round(max(t_batch), 3)],
            "batch_mlups": round(cells / tb / 1e3, 1),
            "seq_ms": round(ts, 3), "seq_ms_spread": [round(min(t_seq), 3), round(max(t_seq), 3)],
            "seq_mlups": round(cells / ts / 1e3, 1),
            "speedup": round(ts / tb, 3), "bit_identical": bool(same)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--grids", default="128x128,128x256,256x256")
    ap.add_argument("--batches", default="1,2,4,8,16,32,64")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=0, help="timesteps per run (0: the grid's shipped step count)")
    ap.add_argument("--warmup", type=int, default=100)
    a = ap.parse_args()
    print(json.dumps({"gpu": gpu_identity(), "tile_rows_knob": os.environ.get("LBM_BATCH_TILE_ROWS"),
                      "thread_rows_knob": os.environ.get("LBM_BATCH_THREAD_ROWS"), "lib": os.path.relpath(L.LIB_PATH, ROOT)}), flush=True)
    ok = True
    for name in a.grids.split(","):
        steps = a.steps or SHIPPED[name][2]
        for b in [int(x) for x in a.batches.split(",")]:
            r = measure(name, b, steps, a.reps, a.warmup)
            ok = ok and r["bit_identical"]
            print(json.dumps(r), flush=True)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
