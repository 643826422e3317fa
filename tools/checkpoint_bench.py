"""Checkpoint rates on one GPU: lbm_gpu_save_rows and lbm_gpu_load_rows against lbm_gpu_download_rows,
and the CLI's checkpoint write and restart times.

Library part: a synthetic N x N channel (walls, 1 % random obstacles, density 0.1, accel 0.005,
omega 1.85) after a few steps, in fp32 and in binary16 storage (LBM_GPU_STORE_F16).  Each call
moves a block of --block rows between the lattice and one pinned host buffer (lbm_gpu_host_alloc);
one pass covers the whole grid (a load pass writes the one buffer into every block: only the rate
counts here).  Per store, after one warm-up pass, --reps passes of save_rows,
load_rows and download_rows, alternating, each timed with a host clock around the blocking calls.
Reported: the median pass time and GB/s of the bytes that cross PCIe (records: 36 B per cell fp32,
18 B binary16; download_rows: 36 B per cell, decoded fp32 for binary16).

CLI part (--cli-n, 0 = skip): the host program on an M x M channel of --cli-steps steps with
LBM_SKIP_FINAL_STATE=1, once with LBM_CHECKPOINT into a temporary directory (its "Elapsed
Checkpoint time" line: digest, save_rows and writing the file, fsync included), then with
LBM_RESTART from that file (its Init time, against the Init time of a run without restart:
reading the file, load_rows and the checksum).  Both are bound by the local disk, not by the GPU.

  python tools/checkpoint_bench.py [--n 16384] [--reps 5] [--cli-n 8192]

Prints the card's name and power limit first, then one JSON line per measurement.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lbm_b200 as L  # noqa: E402
from tools.make_inputs import write_obstacles, write_params  # noqa: E402

D, A, W = 0.1, 0.005, 1.85


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def channel(nx, ny, p=0.01, seed=1):
    m = np.random.default_rng(seed).random((ny, nx), dtype=np.float32) < p
    m[0, :] = m[ny - 1, :] = True
    return m


def bench_library(n, reps, block, steps):
    mask_bits = L.pack_obstacle_bits(channel(n, n))
    for store in ("f32", "f16"):
        flags = L.STORE_F16 if store == "f16" else 0
        with L.Lattice(n, n, D, A, W, obstacles=mask_bits, bits=True, flags=flags) as lat:
            lat.run(steps)
            rec_b = 18 if store == "f16" else 36
            buf = L.PinnedArray((block, n, 9), lat.record_dtype)
            dbuf = L.PinnedArray((block, n, 9), np.float32)
            lib = lat.lib

            def one_pass(kind):
                t0 = time.perf_counter()
                for r0 in range(0, n, block):
                    nr = min(block, n - r0)
                    if kind == "save_rows":
                        rc = lib.lbm_gpu_save_rows(lat.h, r0, nr, buf.array.ctypes.data)
                    elif kind == "load_rows":
                        rc = lib.lbm_gpu_load_rows(lat.h, r0, nr, buf.array.ctypes.data)
                    else:
                        rc = lib.lbm_gpu_download_rows(lat.h, r0, nr, dbuf.array.ctypes.data)
                    if rc != 0:
                        raise L.LbmError(lib.lbm_gpu_last_error().decode())
                return time.perf_counter() - t0

            kinds = ("save_rows", "load_rows", "download_rows")
            for k in kinds:
                one_pass(k)                                  # warm-up
            times = {k: [] for k in kinds}
            for _ in range(reps):
                for k in kinds:
                    times[k].append(one_pass(k))
            for k in kinds:
                t = float(np.median(times[k]))
                nbytes = n * n * (36 if k == "download_rows" else rec_b)
                print(json.dumps({"store": store, "call": k, "n": n, "block_rows": block, "passes": reps,
                                  "median_s": round(t, 4), "min_s": round(min(times[k]), 4),
                                  "max_s": round(max(times[k]), 4), "bytes": nbytes,
                                  "gbs": round(nbytes / t / 1e9, 1)}), flush=True)
            buf.free()
            dbuf.free()


def elapsed(out, what):
    m = re.search(r"Elapsed %s time:\s+([0-9.]+)" % what, out)
    return float(m.group(1)) if m else None


def bench_cli(m, steps, precisions):
    exe = os.path.join(ROOT, "d2q9-bgk")
    with tempfile.TemporaryDirectory() as d:
        params, obst = os.path.join(d, "in.params"), os.path.join(d, "obst.dat")
        write_params(params, m, m, steps, 10, D, A, W)
        write_obstacles(obst, channel(m, m))
        for prec in precisions:
            env = dict(os.environ, LBM_SKIP_FINAL_STATE="1")
            for k in ("LBM_CHECKPOINT", "LBM_CHECKPOINT_EVERY", "LBM_RESTART", "LBM_PRECISION"):
                env.pop(k, None)
            if prec != "f32":
                env["LBM_PRECISION"] = prec
            ckpt = os.path.join(d, "run.ckpt")

            def run(extra):
                r = subprocess.run([exe, params, obst], cwd=d, env=dict(env, **extra), stdout=subprocess.PIPE,
                                   stderr=subprocess.PIPE, text=True)
                if r.returncode != 0:
                    raise RuntimeError(r.stderr)
                return r.stdout

            plain = run({})
            written = run({"LBM_CHECKPOINT": ckpt})
            size = os.path.getsize(ckpt)
            restarted = run({"LBM_RESTART": ckpt})
            w = elapsed(written, "Checkpoint")
            init_plain, init_restart = elapsed(plain, "Init"), elapsed(restarted, "Init")
            print(json.dumps({"cli": prec, "n": m, "steps": steps, "file_bytes": size,
                              "checkpoint_write_s": w, "write_gbs": round(size / w / 1e9, 2) if w else None,
                              "init_s_plain": init_plain, "init_s_restart": init_restart,
                              "restart_load_s": round(init_restart - init_plain, 4),
                              "load_gbs": round(size / (init_restart - init_plain) / 1e9, 2)
                              if init_restart > init_plain else None}), flush=True)
            os.remove(ckpt)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--n", type=int, default=16384)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--block", type=int, default=1024, help="rows per call")
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--cli-n", type=int, default=8192)
    ap.add_argument("--cli-steps", type=int, default=10)
    ap.add_argument("--cli-precisions", default="f32,f16")
    a = ap.parse_args()
    print(json.dumps({"card": card()}), flush=True)
    bench_library(a.n, a.reps, a.block, a.steps)
    if a.cli_n > 0:
        bench_cli(a.cli_n, a.cli_steps, a.cli_precisions.split(","))


if __name__ == "__main__":
    main()
