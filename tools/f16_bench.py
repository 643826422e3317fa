"""MLUPS of shifted binary16 storage (LBM_GPU_STORE_F16) against the fp32 default, on one GPU.

Synthetic channel (1 % random obstacles, d2q9-bgk parameters density 0.1, accel 0.005,
omega 1.85), device time from CUDA events (last_run_device_ms).  The builds alternate within
one process, `--reps` times each, so the spread is the spread of one session.  Also creates one
grid too large for fp32 on this GPU (cells = NULL, LBM_GPU_OBST_BITS), runs it and reports the
mass drift and the digest.

    python tools/f16_bench.py [--grids 4096x4096,8192x8192,16384x16384] [--steps 200] [--reps 3]
                              [--big 32768x81920] [--big-steps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbm_b200 as L  # noqa: E402

D, A, W = 0.1, 0.005, 1.85
KNAME = {L.KERNEL_VEC4: "K1a", L.KERNEL_TB2: "K7", L.KERNEL_TB3: "K10"}
BUILDS = [("fp32 default", 0), ("f16 default", L.STORE_F16), ("f16 K1a-f16", L.STORE_F16 | L.KERNEL_VEC4)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def channel_bits(nx, ny, p=0.01, seed=1):
    """Walls at rows 0 and ny-1 and (p > 0) random obstacles, as LBM_GPU_OBST_BITS words."""
    if p > 0:
        m = np.random.default_rng(seed).random((ny, nx), dtype=np.float32) < p
        m[0, :] = m[ny - 1, :] = True
        return L.pack_obstacle_bits(m)
    bits = np.zeros((ny, (nx + 31) // 32), dtype=np.uint32)
    bits[0, :] = bits[ny - 1, :] = 0xFFFFFFFF
    return bits


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--grids", default="4096x4096,8192x8192,16384x16384")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--big", default="32768x81920")
    ap.add_argument("--big-steps", type=int, default=20)
    a = ap.parse_args()
    print(json.dumps({"card": card()}), flush=True)
    for g in a.grids.split(","):
        nx, ny = map(int, g.split("x"))
        obst = channel_bits(nx, ny)
        lats = [(name, L.Lattice(nx, ny, D, A, W, obstacles=obst, bits=True, flags=f)) for name, f in BUILDS]
        times = {name: [] for name, _ in lats}
        for name, lat in lats:
            lat.run_timed(20)                                      # warm-up
        for _ in range(a.reps):
            for name, lat in lats:
                times[name].append(lat.run_timed(a.steps))
        for name, lat in lats:
            t = np.array(times[name]) * 1e-3
            mlups = nx * ny * a.steps / t / 1e6
            f16 = "f16" in name
            bpu = (18.0 if lat.info().kernel == L.KERNEL_TB2 else 36.0) if f16 else \
                {L.KERNEL_TB2: 36.0, L.KERNEL_TB3: 24.75}.get(lat.info().kernel, 72.0)
            print(json.dumps({"grid": g, "build": name, "kernel": KNAME.get(lat.info().kernel, lat.info().kernel),
                              "mlups_best": round(mlups.max(), 1), "mlups_median": round(float(np.median(mlups)), 1),
                              "spread_pct": round(100 * (mlups.max() - mlups.min()) / mlups.max(), 2),
                              "bytes_per_update": bpu, "achieved_tb_s": round(mlups.max() * 1e6 * bpu / 1e12, 3),
                              "device_gb": round(lat.info().device_bytes / 1e9, 2)}), flush=True)
        for _, lat in lats:
            lat.close()
    if a.big:
        nx, ny = map(int, a.big.split("x"))
        with L.Lattice(nx, ny, D, A, W, obstacles=channel_bits(nx, ny, p=0), bits=True, flags=L.STORE_F16) as lat:
            m0, c0 = lat.digest()
            ms = lat.run_timed(a.big_steps)
            m1, c1 = lat.digest()
            av = lat.av_velocity()
            print(json.dumps({"big_grid": a.big, "fp32_lattice_gb": round(72.0 * nx * ny / 1e9, 1),
                              "device_gb": round(lat.info().device_bytes / 1e9, 1),
                              "kernel": KNAME.get(lat.info().kernel), "steps": a.big_steps,
                              "mlups": round(nx * ny * a.big_steps / (ms * 1e-3) / 1e6, 1),
                              "mass_before": m0, "mass_after": m1, "mass_drift_rel": (m1 - m0) / m0,
                              "checksum": "%016x" % c1, "av_velocity": av}), flush=True)
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
