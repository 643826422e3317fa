#!/usr/bin/env python3
"""Build tuning variants of liblbm_b200.so (same ABI, different compile-time knobs of the
step kernel) into advanced-hpc-lbm_b200/variants/ and, with --run, time each of them on the
16384^2 bench grid (development tool; results go to profiles/r01_kernel_variants.md)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "advanced-hpc-lbm_b200")
OUT = os.path.join(PKG, "variants")
VARIANTS = {
    "base": [],
    "mb6": ["-DLBM_MIN_BLOCKS=6", "-DLBM_PERSIST_MIN_BLOCKS=5"],
    "mb5": ["-DLBM_MIN_BLOCKS=5", "-DLBM_PERSIST_MIN_BLOCKS=4"],
    "mb4": ["-DLBM_MIN_BLOCKS=4", "-DLBM_PERSIST_MIN_BLOCKS=3"],
    "scalar": ["-DLBM_PACKED=0"],
    "scalar_mb5": ["-DLBM_PACKED=0", "-DLBM_MIN_BLOCKS=5", "-DLBM_PERSIST_MIN_BLOCKS=4"],
    "tb2_mb2": ["-DLBM_TB2_THREADS=128", "-DLBM_TB2_MIN_BLOCKS=2"],
    "barrier0": ["-DLBM_BARRIER_MODE=0"],
    "tb2_t128": ["-DLBM_TB2_THREADS=128", "-DLBM_TB2_MIN_BLOCKS=3"],
    "tb2_t64": ["-DLBM_TB2_THREADS=64", "-DLBM_TB2_MIN_BLOCKS=6"],
    "tb3_t64": ["-DLBM_TB2_THREADS=64", "-DLBM_TB3_MIN_BLOCKS=4"],     # K10, 64-thread strips (profiles/r03_k10.md)
    "tb3_mb2": ["-DLBM_TB3_MIN_BLOCKS=2"],                              # K10, 186 registers, 6 warps per SM
    # K10's staging-wait share of its cycles (r07) and the busy fraction of its block slots (r08; run with
    # --kernel tb3, and LBM_GPU_NO_TB3_OVERLAP=1 for passes that do not overlap)
    "tb3_wait": ["-DLBM_EXPERIMENTS"],
}
if os.environ.get("LBM_VARIANTS"):
    VARIANTS = {k: v for k, v in VARIANTS.items() if k in os.environ["LBM_VARIANTS"].split(",")}


def build():
    os.makedirs(OUT, exist_ok=True)
    procs = []
    for name, defs in VARIANTS.items():
        so = os.path.join(OUT, "liblbm_%s.so" % name)
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler",
               "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), *defs,
               os.path.join(PKG, "csrc", "lbm_gpu.cu"), "-o", so]
        procs.append((name, subprocess.Popen(cmd)))
    for name, p in procs:
        assert p.wait() == 0, name


def run():
    for name in VARIANTS:
        env = dict(os.environ, LBM_B200_LIB=os.path.join(OUT, "liblbm_%s.so" % name))
        args = sys.argv[sys.argv.index("--run") + 1:] or ["--steps", "40", "--reps", "3", "--kernel", "vec4"]
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "quick_bench.py"), *args], env=env,
                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        lines = [l for l in r.stdout.splitlines() if "MLUPS" in l]
        best = max(lines, key=lambda l: float(l.split("MLUPS")[0].split()[-1])) if lines else r.stdout[-300:]
        print("%-14s %s" % (name, best), flush=True)


if __name__ == "__main__":
    if "--run" in sys.argv:
        run()
    else:
        build()
