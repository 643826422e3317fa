"""Cost of the obstacle force read-out (lbm_gpu_obstacle_force) against one step of the default kernel.

Cases: the synthetic 16384^2 channel of bench.py (walls, 1 % random obstacles, density 0.1, accel
0.005, omega 1.85) in fp32 and in binary16 storage (LBM_GPU_STORE_F16), and the shipped 1024^2 input.
Each lattice runs a few steps first.  Per case it prints:
  step_ms        device time of one step of the default kernel (lbm_gpu_run over --steps steps, CUDA events)
  call_ms        wall time of the blocking call (whole grid, one box), median / min / max of --reps calls
                 after one warm-up; the calls alternate with the step runs
  kernel_ms      device time of lbm_obstacle_force, median of 3 calls under torch.profiler (CUDA activities)
  solid, links   obstacle cells, and solid cells with at least one fluid neighbour (the cells whose
                 values the kernel reads)
  model_mb       mask bytes plus 16 values per such cell: the least the kernel can read
For the fp32 channel it then times calls with several boxes (kernel and call time as above):
  64 boxes of 64 x 64 cells at random places, 256 such boxes, the whole grid plus 63 small boxes,
  and 256 boxes that tile the grid (16 x 16 boxes of n/16 x n/16): a box costs its own area.
The card's name, power limit and max SM clock are printed at the start and at the end.

  python tools/force_bench.py [--n 16384] [--reps 11] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbm_b200 as L  # noqa: E402

D, A, W = 0.1, 0.005, 1.85


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def channel(nx, ny, p=0.01, seed=1):
    m = np.random.default_rng(seed).random((ny, nx), dtype=np.float32) < p
    m[0, :] = m[ny - 1, :] = True
    return m


def shipped(name):
    lines = open(os.path.join(ROOT, "inputs", "input_%s.params" % name)).read().split()
    nx, ny = int(lines[0]), int(lines[1])
    m = np.zeros((ny, nx), dtype=bool)
    for line in open(os.path.join(ROOT, "inputs", "obstacles_%s.dat" % name)):
        if line.strip():
            x, y, _ = map(int, line.split())
            m[y, x] = True
    return m, float(lines[4]), float(lines[5]), float(lines[6])


def link_cells(m):
    """solid cells with a fluid neighbour along one of the 8 speeds (periodic)"""
    fluid_nb = np.zeros_like(m)
    for dx, dy in ((1, 0), (0, 1), (-1, 0), (0, -1), (1, 1), (-1, 1), (-1, -1), (1, -1)):
        fluid_nb |= ~np.roll(m, shift=(-dy, -dx), axis=(0, 1))
    return int((m & fluid_nb).sum())


def kernel_ms(lat, out_dir, tag, boxes=None):
    import torch
    from torch.profiler import ProfilerActivity, profile
    runs = []
    for rep in range(3):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            lat.obstacle_force(boxes)
        path = os.path.join(out_dir, "trace_force_%s_%d.json" % (tag, rep))
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
        runs.append(sum(e["dur"] for e in ev if e.get("cat") == "kernel" and "lbm_obstacle_force" in e["name"]) * 1e-3)
    torch.cuda.synchronize()
    return sorted(runs)[1], runs


def measure(tag, m, density, accel, omega, flags, a):
    ny, nx = m.shape
    elem = 2 if flags & L.STORE_F16 else 4
    solid, links = int(m.sum()), link_cells(m)
    with L.Lattice(nx, ny, density, accel, omega, obstacles=L.pack_obstacle_bits(m), bits=True, flags=flags) as lat:
        lat.run_timed(a.steps)                               # warm-up of the step kernel
        lat.obstacle_force()                                 # ... and of the read-out
        steps, calls = [], []
        for _ in range(a.reps):
            steps.append(lat.run_timed(a.steps) / a.steps)
            t0 = time.perf_counter()
            lat.obstacle_force()
            calls.append((time.perf_counter() - t0) * 1e3)
        k_med, k_all = kernel_ms(lat, a.out, tag)
        info = lat.info()
        if tag.endswith("_f32") and nx == a.n:
            box_cases(lat, a)
    c = np.array(calls)
    print(json.dumps({"case": tag, "nx": nx, "ny": ny, "kernel_choice": info.kernel,
                      "step_ms": round(float(np.median(steps)), 4),
                      "call_ms_median": round(float(np.median(c)), 4), "call_ms_min": round(float(c.min()), 4),
                      "call_ms_max": round(float(c.max()), 4),
                      "kernel_ms": round(k_med, 4), "kernel_ms_of_3_calls": [round(r, 4) for r in k_all],
                      "call_over_step": round(float(np.median(c)) / float(np.median(steps)), 3),
                      "solid": solid, "links": links,
                      "model_mb": round((nx * ny / 8 + links * 16 * elem) / 1e6, 1)}), flush=True)


def box_cases(lat, a):
    n = a.n
    rng = np.random.default_rng(2)

    def small(k):
        x0, y0 = rng.integers(0, n - 64, k), rng.integers(0, n - 64, k)
        return np.stack([x0, y0, x0 + 64, y0 + 64], axis=1)
    t = n // 16
    tiles = np.array([(i * t, j * t, (i + 1) * t, (j + 1) * t) for j in range(16) for i in range(16)])
    cases = [("64 boxes of 64x64", small(64)), ("256 boxes of 64x64", small(256)),
             ("whole grid + 63 boxes of 64x64", np.concatenate([[(0, 0, n, n)], small(63)])),
             ("256 boxes tiling the grid", tiles)]
    for name, b in cases:
        b = np.ascontiguousarray(b, dtype=np.int32)
        lat.obstacle_force(b)                                # warm-up
        calls = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            lat.obstacle_force(b)
            calls.append((time.perf_counter() - t0) * 1e3)
        k_med, k_all = kernel_ms(lat, a.out, "boxes", b)
        print(json.dumps({"case": "channel_%d_f32" % n, "boxes": name, "n_boxes": len(b),
                          "cells_in_boxes": int(np.sum((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1]))),
                          "call_ms_median": round(float(np.median(calls)), 4), "kernel_ms": round(k_med, 4),
                          "kernel_ms_of_3_calls": [round(r, 4) for r in k_all]}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default=None, help="directory for the profiler traces (default: a new temporary one)")
    a = ap.parse_args()
    a.out = a.out or tempfile.mkdtemp(prefix="force_bench_")
    os.makedirs(a.out, exist_ok=True)
    print(json.dumps({"card": card()}), flush=True)
    m = channel(a.n, a.n)
    measure("channel_%d_f32" % a.n, m, D, A, W, 0, a)
    measure("channel_%d_f16" % a.n, m, D, A, W, L.STORE_F16, a)
    del m
    m, d, acc, om = shipped("1024x1024")
    measure("shipped_1024x1024_f32", m, d, acc, om, 0, a)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
