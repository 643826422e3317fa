"""Snapshot read-outs on one GPU: lbm_gpu_final_fields against lbm_gpu_coarse_fields.

Synthetic 16384^2 channel (walls, 1 % random obstacles, density 0.1, accel 0.005, omega 1.85)
after a few steps, in fp32 and in binary16 storage (LBM_GPU_STORE_F16).  Output buffers come
from lbm_gpu_host_alloc (pinned).  Cases: final_fields; coarse_fields factor 1 / F16, and
factors 4, 8, 16 in F32 and F16.

  python tools/coarse_fields_bench.py [--n 16384] [--reps 7]            wall time of the blocking call
  python tools/coarse_fields_bench.py --profile DIR [--n 16384]         kernel time (torch.profiler)

The default mode prints, per case, the median and spread of the wall time of the blocking call
over --reps calls after one warm-up call, and the bytes it sends to the host.  --profile, in a
process of its own, records three calls of each case with torch.profiler (CUDA activities), one
per trace under DIR, and prints for the median call the summed device time of the read-out
kernels, the lattice bytes they read per second and that rate's share of the measured copy
bandwidth: MEASURED_PEAKS.json hbm_gbs where the file exists, else a device-to-device copy timed
in the same process.  Both modes print the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbm_b200 as L  # noqa: E402

D, A, W = 0.1, 0.005, 1.85
CASES = [("final_fields", 0, False), ("coarse f1 F16", 1, True),
         ("coarse f4 F32", 4, False), ("coarse f4 F16", 4, True),
         ("coarse f8 F32", 8, False), ("coarse f8 F16", 8, True),
         ("coarse f16 F32", 16, False), ("coarse f16 F16", 16, True)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def channel_bits(nx, ny, p=0.01, seed=1):
    m = np.random.default_rng(seed).random((ny, nx), dtype=np.float32) < p
    m[0, :] = m[ny - 1, :] = True
    return L.pack_obstacle_bits(m)


def buffers(lat, factor, f16):
    """Pinned outputs of one case (kept for the whole run)."""
    if factor == 0:
        shape, dt = (lat.ny, lat.nx), np.float32
    else:
        shape, dt = (-(-lat.ny // factor), -(-lat.nx // factor)), (np.float16 if f16 else np.float32)
    return [L.PinnedArray(shape, dt) for _ in range(4)]


def call(lat, factor, f16, bufs):
    out = [b.array for b in bufs]
    if factor == 0:
        lat.final_fields(out=out)
    else:
        lat.coarse_fields(factor, f16=f16, out=out)


def lattice_bytes(nx, ny, store):
    """What a read-out kernel has to read: nine planes and the bit mask."""
    return nx * ny * (18 if store == "f16" else 36) + nx * ny // 8


def copy_gbs():
    """Device-to-device copy bandwidth, (read + write) bytes per second, median of 20 copies of 2 GiB."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    import torch
    a = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    ts = []
    for _ in range(20):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e-3)
    del a, b
    return 2 * (1 << 31) / float(np.median(ts)) / 1e9, "device-to-device copy of 2 GiB, this process"


def kernel_ms(trace_path):
    """Summed device time of the read-out kernels in a chrome trace, and their count."""
    with open(trace_path) as f:
        ev = json.load(f)["traceEvents"]
    ks = [e for e in ev if e.get("cat") == "kernel" and ("lbm_coarse_fields" in e["name"] or "lbm_fields" in e["name"])]
    return sum(e["dur"] for e in ks) * 1e-3, len(ks)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--stores", default="f32,f16")
    ap.add_argument("--profile", default=None, help="directory for the torch.profiler traces")
    a = ap.parse_args()
    print(json.dumps({"card": card()}), flush=True)
    nx = ny = a.n
    peak = None
    if a.profile:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        peak, peak_src = copy_gbs()
        print(json.dumps({"hbm_gbs": round(peak, 1), "source": peak_src}), flush=True)
        os.makedirs(a.profile, exist_ok=True)
    for store in a.stores.split(","):
        flags = L.STORE_F16 if store == "f16" else 0
        with L.Lattice(nx, ny, D, A, W, obstacles=channel_bits(nx, ny), bits=True, flags=flags) as lat:
            lat.run_timed(a.steps)
            bufs = {name: buffers(lat, f, h) for name, f, h in CASES}
            for name, f, h in CASES:
                call(lat, f, h, bufs[name])                       # warm-up
            if a.profile:
                for name, f, h in CASES:
                    runs = []
                    for rep in range(3):                          # one profiled call each
                        with profile(activities=[ProfilerActivity.CUDA]) as prof:
                            call(lat, f, h, bufs[name])
                        path = os.path.join(a.profile, "trace_%s_%s_%d.json" % (store, name.replace(" ", "_"), rep))
                        prof.export_chrome_trace(path)
                        runs.append(kernel_ms(path))
                    ms, n = sorted(runs)[1]                        # the median call
                    rate = lattice_bytes(nx, ny, store) / (ms * 1e-3) / 1e9
                    print(json.dumps({"store": store, "case": name, "kernel_ms": round(ms, 3), "kernels": n,
                                      "kernel_ms_of_3_calls": [round(r[0], 3) for r in runs],
                                      "lattice_gb": round(lattice_bytes(nx, ny, store) / 1e9, 3),
                                      "read_gbs": round(rate, 1), "share_of_hbm_gbs": round(rate / peak, 3)}),
                          flush=True)
            else:
                times = {name: [] for name, _, _ in CASES}
                for _ in range(a.reps):                           # cases alternate within each repeat
                    for name, f, h in CASES:
                        t0 = time.perf_counter()
                        call(lat, f, h, bufs[name])
                        times[name].append((time.perf_counter() - t0) * 1e3)
                for name, f, h in CASES:
                    t = np.array(times[name])
                    sent = sum(b.array.nbytes for b in bufs[name])
                    print(json.dumps({"store": store, "case": name, "wall_ms_median": round(float(np.median(t)), 2),
                                      "wall_ms_min": round(float(t.min()), 2), "wall_ms_max": round(float(t.max()), 2),
                                      "d2h_mb": round(sent / 1e6, 1),
                                      "d2h_gbs": round(sent / (float(np.median(t)) * 1e-3) / 1e9, 1)}), flush=True)
            for bl in bufs.values():
                for b in bl:
                    b.free()
    print(json.dumps({"card": card()}), flush=True)


if __name__ == "__main__":
    main()
