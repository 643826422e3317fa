#!/usr/bin/env python3
"""bench.py -- headline benchmark of the d2q9-bgk timestep loop on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--timesteps T] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): MLUPS = lattice-cell updates per second / 1e6, and the achieved
HBM bandwidth it implies (72 B per update) against the measured B200 peak.

Workload: the synthetic channel of BASELINE.json configs[3]/[4] -- nx = 16384, ny = 16384
rows per GPU (weak scaling), walls on rows 0 and ny-1, Bernoulli(1 %) obstacles, rest
state at t = 0.  One bench "step" is one pass of the step loop: T consecutive timesteps
(`--timesteps`, default 200, the lower end of SURVEY.md section 8d's 200-1000) issued by
one lbm_gpu_run() call.  The lattice (19.3 GB per GPU) is far larger than L2 (126 MB),
so nothing stays cached between timesteps or steps.

  value   lattice resident in HBM, K steps timed with CUDA events on the library's
          stream (max over ranks): all cells x T x K / time.
  e2e     the same K steps through the C-ABI from HOST buffers, everything inside the
          timed region every step: lbm_gpu_create (pinned int32 obstacle array -> HBM,
          like the reference's int obstacles[]), lbm_gpu_run (T timesteps, av_vels to
          the host), lbm_gpu_final_fields (u_x,u_y,|u|,pressure of every cell -> pinned
          host arrays, what write_values needs), lbm_gpu_destroy.
  --impl reference   the reference's own timestep_new2, compiled from /root/reference
          into oracle/_ref (or the oracle port if that is absent), on the host cores
          with all threads, on a bounded sample of the same workload.

Also in the JSON line (round 2):
  parity    run BEFORE the timed region: the kernels of the headline path (K1a and the
            two-timestep K7, MULTI=true instantiations when N > 1, through create_slab /
            IPC / connect_all / run_sums) against the CPU oracle's exact lattice checksum and
            av_vels (strict build) and against a one-slab GPU run (default build); at N > 1
            also the protocol-exit test (a rank asked for fewer steps makes the others return
            an error within the time-out); total-mass drift of the full grid over the timed
            timesteps.  A mismatch makes the process exit non-zero.
  strong    N > 1: the single 16384 x 16384 grid split over the N GPUs (configs[3]),
            2 x T timesteps, device-timed, max over ranks.
  shipped   N = 1: the reference's four shipped inputs, full step counts: MLUPS, kernel
            chosen, check.py's criterion against the golden files.
  roofline  of the dominant kernel; K7 advances TWO timesteps per launch with the 72 B per
            cell of one pass, so algorithmic bytes per update = 36; `traffic` is the ncu
            figure of the committed capture named in `traffic_source`.

--dump-outputs DIR writes what the last timed step of `value` computed, so that two builds
can be compared output for output on the same inputs (the workload is seeded):
  av_vels.npy           float32 (T,), the step's av_vels as lbm_gpu_run returns them
  cells_rows.npy        float32 (64, nx, 9), lattice rows after the step (lbm_gpu_download layout)
  cells_rows_index.npy  float64 (64,), which rows: a fixed seeded sample of the grid
About 38 MB at nx = 16384.  The last timed step then fetches its av_vels (one small kernel
after the step's end event: the device time is unchanged, `gpu_launches` counts it).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only: no __pycache__ written into it

from tools.make_inputs import channel_mask  # noqa: E402

# LBM_BENCH_NX / LBM_BENCH_ROWS shrink the grid for the harness's own tests; the benchmark
# contract is the default 16384 x 16384 per GPU.
NX = int(os.environ.get("LBM_BENCH_NX", "16384"))
ROWS_PER_GPU = int(os.environ.get("LBM_BENCH_ROWS", "16384"))
DENSITY, ACCEL, OMEGA = 0.1, 0.005, 1.85
BYTES_PER_UPDATE = 72.0            # 9 fp32 loads + 9 fp32 stores (SURVEY.md section 8d)
CPU_SAMPLE_ROWS = min(1024, ROWS_PER_GPU)   # CPU legs run a 16384 x 1024 slab of the same generator
HBM_FALLBACK_GBS = 6650.0          # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_ROWS, DUMP_SEED = 64, 20240229          # --dump-outputs: lattice rows sampled, and their seed


# ------------------------------------------------------------------------- clocks ----
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # samples under load: power above 40 % of the observed maximum
        if sm:
            pmax = max(power)
            load = [s for s, p in zip(sm, power) if p >= 0.4 * pmax] or sm
            return {"sm_mhz": float(np.median(load)), "sm_max_mhz": max(mx), "power_w_max": pmax,
                    "samples": len(sm), "reasons": sorted(reasons)}
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except (OSError, KeyError, ValueError):
        return HBM_FALLBACK_GBS, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def ncu_traffic(kernel):
    """dram bytes per launch of the dominant kernel, from the committed `ncu --set full` capture
    of the same kernel at the same size (profiles/): never measured inside a bench run, because
    a number taken under a profiler is not a bench value -- hence the source label."""
    name = "r02_ncu_tb2_summary.json" if kernel == 512 else "ncu_step_kernel_summary.json"
    p = os.path.join(ROOT, "profiles", name)
    try:
        with open(p) as f:
            d = json.load(f)
        return {"dram_bytes_per_launch": d.get("dram_bytes_per_launch"),
                "source": "profiles/%s (ncu --set full, library %s)" % (name, d.get("library_sha256_16", "of round 1"))}
    except (OSError, ValueError):
        return {"dram_bytes_per_launch": None, "source": "no committed ncu capture for this kernel"}


# ----------------------------------------------------------------- CPU reference ----
class RefParam(ctypes.Structure):      # t_param of the reference, d2q9-bgk.c:64-73
    _fields_ = [("nx", ctypes.c_int), ("ny", ctypes.c_int), ("maxIters", ctypes.c_int),
                ("reynolds_dim", ctypes.c_int), ("density", ctypes.c_float), ("accel", ctypes.c_float),
                ("omega", ctypes.c_float)]


def cpu_reference_mlups(budget_s, threads=None, prefer="omp"):
    """Time the reference's own timestep_new2 (d2q9-bgk.c:228) on a 16384 x 1024 slab of the
    bench workload for about budget_s seconds.  Uses oracle/_ref (the reference compiled
    from /root/reference by oracle/build_oracle.py); falls back to the oracle port.
    This is the one place outside tests/ that executes anything under oracle/: it is the
    measured CPU baseline, never part of the GPU path."""
    nx, ny = NX, CPU_SAMPLE_ROWS
    ncores = os.cpu_count() or 1
    threads = threads or ncores
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    kind = "reference"
    lib = None
    name = "libref_f32_omp.so" if (prefer == "omp" and threads > 1) else "libref_f32_fast.so"
    if os.path.exists(os.path.join(ref_dir, name)):
        lib = ctypes.CDLL(os.path.join(ref_dir, name))
        fn = lib.timestep_new2
        fn.argtypes = [RefParam, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        fn.restype = ctypes.c_float
        prm = RefParam(nx, ny, 1, 10, DENSITY, ACCEL, OMEGA)
        step = lambda a, b, o: fn(prm, a, b, o)
        if name == "libref_f32_fast.so":
            threads = 1
    else:
        kind = "port"
        so = os.path.join(ROOT, "oracle", "liblbm_oracle.so")
        if not os.path.exists(so):
            subprocess.check_call([sys.executable, os.path.join(ROOT, "oracle", "build_oracle.py")])
        lib = ctypes.CDLL(so)
        fn = lib.oracle_timestep_f32
        fl = ctypes.c_float
        fn.argtypes = [ctypes.c_int, ctypes.c_int, fl, fl, fl] + [ctypes.c_void_p] * 5
        fn.restype = fl
        scratch = np.empty(nx * ny, dtype=np.float32)
        step = lambda a, b, o: fn(nx, ny, DENSITY, ACCEL, OMEGA, a, b, o, scratch.ctypes.data, None)
    mask = channel_mask(nx, ny).astype(np.int32)
    w = (np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4) * DENSITY).astype(np.float32)
    a = np.tile(w, (ny * nx, 1))
    b = np.empty_like(a)
    pa, pb, po = a.ctypes.data, b.ctypes.data, mask.ctypes.data
    step(pa, pb, po)                      # warm-up (page faults of b)
    pa, pb = pb, pa
    n, t0 = 0, time.perf_counter()
    while True:
        step(pa, pb, po)
        pa, pb = pb, pa
        n += 1
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 10000:
            break
    return {"value": nx * ny * n / dt / 1e6, "unit": "MLUPS", "cores": int(threads), "kind": kind,
            "sample": "%dx%d slab of the same channel generator, %d timesteps of timestep_new2 in %.1f s "
                      "(%s)" % (nx, ny, n, dt, name if kind == "reference" else "oracle port"),
            "host_cores_visible": ncores}, n, dt


def run_reference_arm(args, rank, world):
    if rank != 0:
        return 0
    per_step_budget = max(2.0, min(20.0, 90.0 / max(1, args.steps + args.warmup)))
    if os.environ.get("LBM_BENCH_CPU_BUDGET_S"):          # tests: shorter CPU sample
        per_step_budget = float(os.environ["LBM_BENCH_CPU_BUDGET_S"])
    for _ in range(args.warmup):
        cpu_reference_mlups(per_step_budget / 4)
    vals, tot_updates, tot_time = [], 0.0, 0.0
    info = None
    for _ in range(args.steps):
        info, n, dt = cpu_reference_mlups(per_step_budget)
        tot_updates += NX * CPU_SAMPLE_ROWS * n
        tot_time += dt
    value = tot_updates / tot_time / 1e6
    info["value"] = value
    line = {
        "impl": "reference", "metric": "MLUPS (d2q9-bgk lattice updates per second / 1e6)",
        "value": value, "unit": "MLUPS", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_time / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, world),
                       cpu_arm="timestep_new2 of the reference (OpenMP-annotated build, one pragma before the row loop "
                               "d2q9-bgk.c:787) timed on a %dx%d SLAB SAMPLE of the workload's generator, not the whole "
                               "grid; MLUPS does not depend on the grid height" % (NX, CPU_SAMPLE_ROWS)),
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": "MLUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(args, world):
    ny = ROWS_PER_GPU * world if args.scaling == "weak" else ROWS_PER_GPU
    return {"workload": "synthetic %dx%d channel (walls rows 0 and ny-1, Bernoulli 1%% obstacles, seed 20240229), "
                        "%d rows per GPU" % (NX, ny, ny // world),
            "nx": NX, "ny": ny, "timesteps_per_step": args.timesteps,
            "density": DENSITY, "accel": ACCEL, "omega": OMEGA,
            "l2": "inputs larger than L2 (%.1f GB lattice per GPU vs 126 MB), no flush needed"
                  % (NX * (ny // world) * 72 / 1e9),
            "parallelism": "row slabs, %d GPU(s), halo rows pushed by the step kernel over NVLink" % world}


# ------------------------------------------------------------------------ GPU arm ----
class Ranks:
    """torch.distributed plumbing of the N > 1 launch: barriers and small reductions only."""

    def __init__(self, rank, local_rank, world):
        self.rank, self.local_rank, self.world = rank, local_rank, world
        self.dist = None
        if world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def _reduce(self, values, op, dtype):
        if self.dist is None:
            return list(values)
        import torch
        t = torch.tensor(list(values), dtype=dtype, device="cuda")
        self.dist.all_reduce(t, op=op)
        return t.cpu().tolist()

    def max(self, x):
        return x if self.dist is None else float(self._reduce([x], self.dist.ReduceOp.MAX, _f64())[0])

    def sum(self, x):
        return x if self.dist is None else float(self._reduce([x], self.dist.ReduceOp.SUM, _f64())[0])

    def sum_array(self, a):
        a = np.asarray(a, dtype=np.float64)
        return a if self.dist is None else np.array(self._reduce(a, self.dist.ReduceOp.SUM, _f64()))

    def sum_f32_array(self, a):
        """element-wise float32 sum over ranks, through the GPU (for arrays too big for sum_array)"""
        if self.dist is None:
            return a
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.cpu().numpy()

    def sum_u64(self, x):
        """wrapping 64-bit sum over ranks (16-bit pieces in int64, so nothing overflows on the way)"""
        if self.dist is None:
            return int(x) & (2 ** 64 - 1)
        import torch
        pieces = [(int(x) >> (16 * i)) & 0xffff for i in range(4)]
        tot = self._reduce(pieces, self.dist.ReduceOp.SUM, torch.int64)
        return sum(int(v) << (16 * i) for i, v in enumerate(tot)) & (2 ** 64 - 1)

    def all_true(self, ok):
        return bool(ok) if self.dist is None else self.sum(0.0 if ok else 1.0) == 0.0

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def _f64():
    import torch
    return torch.float64


def bind_near_gpu(local_rank):
    """N > 1: keep this rank on the CPU cores next to its GPU (sysfs local_cpulist of the GPU's
    PCI device), as an MPI launcher would.  The page-locked host buffers of the end-to-end
    leg are then allocated on that NUMA node and eight GPUs do not push 43 GB per step
    through one socket's memory.  LBM_BENCH_BIND=0 switches it off."""
    if os.environ.get("LBM_BENCH_BIND", "1") == "0":
        return "off"
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30)
        bus = r.stdout.strip().lower()[-12:]
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no usable cores in " + spec
        os.sched_setaffinity(0, cpus)
        return "cores " + spec
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        return "unavailable (%s)" % type(e).__name__


KERNEL_NAMES = {4: "lbm_step_scalar", 16: "lbm_step_vec4", 64: "lbm_steps_persistent", 8: "lbm_step_tma",
                256: "lbm_steps_cluster", 2048: "lbm_steps_pairs (two timesteps per grid barrier)", 512: "lbm_step2_tb (two timesteps per pass) + lbm_step_vec4 for an odd step"}


def connect(lat, L, slabs, R):
    """wire a slab handle to its neighbours through the real IPC path, all ranks' descriptors"""
    lat.ipc_connect_all(slabs.gather_descriptors(lat.ipc_export(), R.world, R.dist))
    R.barrier()
    lat.ipc_prepare()
    R.barrier()


def parity_leg(L, slabs, R):
    """Driver-visible proof that the path the timed region uses is CORRECT, run before it.

    N > 1: every rank builds its rows of a small uneven grid (random lattice, 2 % obstacles,
    obstacles on the wrap edges and on the accelerated row ny-2) and runs 25 timesteps in two
    calls through lbm_gpu_create_slab -> ipc_export / connect_all / prepare -> run_sums, i.e.
    the MULTI=true kernels, peer stores, device flags and CUDA IPC of the headline run.  The
    LBM_GPU_STRICT build must reproduce the CPU oracle's lattice (exact checksum over all
    speeds) and its av_vels; the default build must reproduce a one-slab GPU run bit for bit.
    Done for a ragged width (one-step kernel) and for a width the two-step kernel takes.
    N = 1: the same comparison for the single-GPU instantiations.
    The oracle (tests/oracle_lib.py -> oracle/) is used here as the checker only."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    world, rank = R.world, R.rank
    D, A, W = DENSITY, ACCEL, OMEGA
    ny, steps, first = 67 * world + 3, 25, 9
    out = {"checked": True, "ok": True, "ranks": world, "grid_rows": ny, "timesteps": steps, "cases": []}

    def fail(msg):
        out["ok"] = False
        out.setdefault("errors", []).append(msg)

    def run_slabs(nx, cells, obst, flags):
        r0, k = L.split_rows(ny, world)[rank]
        if world == 1:
            lat = L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=flags)
        else:
            lat = L.Lattice(nx, ny, D, A, W, cells=cells[r0:r0 + k], obstacles=obst[r0:r0 + k], slab=(r0, k),
                            device_ids=[R.local_rank], flags=flags)
            connect(lat, L, slabs, R)
        sums = np.concatenate([lat.run_sums(first), lat.run_sums(steps - first)])
        _, cs = lat.digest()
        info = lat.info()
        lat.close()
        return R.sum_array(sums), R.sum_u64(cs), R.sum(float(info.local_free_cells)), int(info.kernel)

    # the two kernels of the headline path, named explicitly (a grid this small would otherwise
    # take the L2-resident persistent kernel on one GPU): K1a for a ragged width, K7 otherwise
    for nx, want in ((515, L.KERNEL_VEC4), (1024, L.KERNEL_TB2)):
        cells, obst = O.random_lattice(nx, ny, seed=1000 + nx + world, p_obst=0.02)
        obst[ny - 2, ::7] = 1
        case = {"nx": nx, "ny": ny}
        try:
            sums, cs, free, kern = run_slabs(nx, cells, obst, L.STRICT | want)
            case["kernel"] = "%s<float, STRICT, MULTI=%s>" % (KERNEL_NAMES.get(kern, str(kern)), "true" if world > 1 else "false")
            if kern != want:
                fail("nx=%d: expected kernel %d, the library chose %d" % (nx, want, kern))
            fsums, fcs, _, _ = run_slabs(nx, cells, obst, want)
            if rank == 0:
                ref, _, av_ref = O.run(cells, obst, steps, D, A, W)
                case["checksum"] = "%016x" % cs
                case["oracle_checksum"] = "%016x" % L.lattice_checksum(ref)
                case["strict_lattice_equals_oracle"] = case["checksum"] == case["oracle_checksum"]
                case["strict_av_vels_max_rel_err"] = float(np.max(np.abs(sums / free - av_ref) / np.abs(av_ref)))
                with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_VEC4) as one:
                    s1 = np.concatenate([one.run_sums(first), one.run_sums(steps - first)])
                    case["strict_equals_one_slab"] = (one.digest()[1] == cs) and bool(np.allclose(s1, sums, rtol=1e-12, atol=0))
                with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.KERNEL_VEC4) as one:
                    s1 = np.concatenate([one.run_sums(first), one.run_sums(steps - first)])
                    case["default_build_equals_one_slab"] = (one.digest()[1] == fcs) and bool(np.allclose(s1, fsums, rtol=1e-12, atol=0))
                if not (case["strict_lattice_equals_oracle"] and case["strict_av_vels_max_rel_err"] < 1e-9 and
                        case["strict_equals_one_slab"] and case["default_build_equals_one_slab"]):
                    fail("nx=%d: mismatch %r" % (nx, case))
        except Exception as e:       # a library error is a parity failure too
            fail("nx=%d: %s: %s" % (nx, type(e).__name__, e))
        out["cases"].append(case)

    if world > 1:
        # the flag protocol has an exit: rank 1 is asked for fewer steps, the others must come
        # back with an error within the time-out instead of spinning inside a kernel
        saved = os.environ.get("LBM_GPU_SYNC_TIMEOUT_MS")
        os.environ["LBM_GPU_SYNC_TIMEOUT_MS"] = "1500"
        try:
            nx = 1024
            cells, obst = O.random_lattice(nx, ny, seed=77, p_obst=0.02)
            r0, k = L.split_rows(ny, world)[rank]
            lat = L.Lattice(nx, ny, D, A, W, cells=cells[r0:r0 + k], obstacles=obst[r0:r0 + k], slab=(r0, k),
                            device_ids=[R.local_rank])
            connect(lat, L, slabs, R)
            t0 = time.perf_counter()
            good = True
            try:
                lat.run_sums(4 if rank == 1 else 24)
                good = (rank == 1)
            except L.LbmError as e:
                good = (rank != 1) and "abandoned" in str(e)
            secs = R.max(time.perf_counter() - t0)
            R.barrier()
            lat.close()
            out["protocol_exit"] = {"ok": R.all_true(good), "seconds": secs, "timeout_ms": 1500}
            if not out["protocol_exit"]["ok"] or secs > 30:
                fail("protocol exit: a rank hung or returned no error (%.1f s)" % secs)
        except Exception as e:
            fail("protocol exit: %s: %s" % (type(e).__name__, e))
        finally:
            if saved is None:
                del os.environ["LBM_GPU_SYNC_TIMEOUT_MS"]
            else:
                os.environ["LBM_GPU_SYNC_TIMEOUT_MS"] = saved
    out["ok"] = R.all_true(out["ok"])
    return out


def shipped_block(L):
    """BASELINE.json configs 1-3: the reference's four shipped inputs, full step counts, on one
    GPU through the C-ABI.  Device MLUPS, the kernel the library chose, and the verdict of
    check/check.py's criterion (worst |100 (ref - sim) / sim| of av_vels and of the final
    pressure field against the golden files, 1 % tolerance) evaluated on the arrays."""
    from tools.make_inputs import SHIPPED, shipped_mask
    res = {}
    for name, (nx, ny, iters, _re, density, accel, omega, _rows, _cols) in SHIPPED.items():
        gold = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        mask = shipped_mask(name).astype(np.int32)
        with L.Lattice(nx, ny, density, accel, omega, obstacles=mask, max_iters=iters) as lat:
            lat.run_timed(min(iters, 2000))                      # warm-up; then the full run from the rest state
        with L.Lattice(nx, ny, density, accel, omega, obstacles=mask, max_iters=iters) as lat:
            av = lat.run(iters)
            info = lat.info()
            ms = info.last_run_device_ms
            pressure = lat.final_fields()[3]
        d_av = float(np.max(np.abs(100.0 * (gold["av_vels"] - av) / av)))
        d_p = float(np.max(np.abs(100.0 * (gold["pressure"] - pressure) / pressure)))
        res[name] = {"mlups": nx * ny * iters / (ms * 1e-3) / 1e6, "us_per_timestep": 1e3 * ms / iters,
                     "timesteps": iters, "kernel": KERNEL_NAMES.get(int(info.kernel), str(info.kernel)),
                     "av_vels_max_pct_vs_golden": d_av, "pressure_max_pct_vs_golden": d_p,
                     "check": "pass" if (np.isfinite(d_av) and np.isfinite(d_p) and d_av <= 1.0 and d_p <= 1.0) else "FAIL"}
    return res


def dump_outputs(path, lat, R, sums, ny, row0, nrows):
    """--dump-outputs: the av_vels of the last timed step and a seeded sample of lattice rows
    after it.  Each rank downloads the sampled rows it holds; rank 0 writes the files."""
    free = R.sum(float(lat.info().local_free_cells))
    av = (R.sum_array(sums) / free).astype(np.float32)        # lbm_gpu_run's own rounding
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(ny, size=min(DUMP_ROWS, ny), replace=False))
    cells = np.zeros((rows.size, NX, 9), dtype=np.float32)
    for i, r in enumerate(rows):
        if row0 <= r < row0 + nrows:
            cells[i] = lat.download_rows(int(r), 1)[0]
    cells = R.sum_f32_array(cells)          # each row is held by one rank, the others add zeros
    if R.rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "av_vels.npy"), av)
        np.save(os.path.join(path, "cells_rows.npy"), cells)
        np.save(os.path.join(path, "cells_rows_index.npy"), rows.astype(np.float64))


def library_id(L):
    import hashlib
    with open(L.LIB_PATH, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--timesteps", type=int, default=200, help="lattice timesteps per bench step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 16384 rows per GPU (default, the contract); strong: 16384 rows in total "
                         "(BASELINE.json configs[3])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-shipped", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU arm (--impl b200)")
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step (--steps >= 1)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3                      # timing rule: at least 3 warm-up steps

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.exit("bench.py --gpus %d must be launched with torch.distributed.run --nproc-per-node %d"
                     % (args.gpus, args.gpus))
        args.gpus = world

    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    binding = bind_near_gpu(local_rank) if world > 1 else "not needed (1 GPU)"
    import lbm_b200 as L
    slabs = __import__("importlib").import_module("advanced-hpc-lbm_b200.slabs")
    R = Ranks(rank, local_rank, world)
    barrier, max_over_ranks, sum_over_ranks = R.barrier, R.max, R.sum

    # ---- parity first: a fast wrong answer is not a result -----------------------------
    parity = {"checked": False}
    if not args.no_parity:
        parity = parity_leg(L, slabs, R)

    T, K, W = args.timesteps, args.steps, args.warmup

    # host arrays: page-locked (ordinary memory if the box refuses to pin that much)
    host_memory = "pinned"

    class _Pageable:
        def __init__(self, shape, dtype):
            self.array = np.empty(shape, dtype=dtype)

        def free(self):
            self.array = None

    def host_array(shape, dtype):
        nonlocal host_memory
        try:
            return L.PinnedArray(shape, dtype)
        except L.LbmError:
            host_memory = "pageable"
            return _Pageable(shape, dtype)

    def make_lattice(ny, row0, nrows, obstacles, bits=False):
        # LBM_GPU_POOL: device memory of a destroyed lattice is reused by the next create
        if world == 1:
            return L.Lattice(NX, ny, DENSITY, ACCEL, OMEGA, obstacles=obstacles, bits=bits, flags=L.POOL)
        lat = L.Lattice(NX, ny, DENSITY, ACCEL, OMEGA, obstacles=obstacles, bits=bits, slab=(row0, nrows),
                        device_ids=[local_rank], flags=L.POOL)
        connect(lat, L, slabs, R)
        return lat

    def timed_runs(lat, n_runs, warm, last_sums=None):
        for _ in range(warm):
            lat.run_timed(T)
        barrier()
        t0 = time.perf_counter()
        dev_ms = 0.0
        for i in range(n_runs):
            if last_sums is not None and i == n_runs - 1:
                last_sums[...] = lat.run_sums(T)     # same device-timed step, av_vels sums fetched after it
                dev_ms += lat.info().last_run_device_ms
            else:
                dev_ms += lat.run_timed(T)          # returns with the device idle (stream sync inside)
        barrier()
        return max_over_ranks(dev_ms), max_over_ranks(time.perf_counter() - t0)

    # ---- value: lattice resident, device-timed ------------------------------------
    ny = ROWS_PER_GPU * world if args.scaling == "weak" else ROWS_PER_GPU
    row0, nrows = L.split_rows(ny, world)[rank]
    cells_total = float(NX) * float(ny)
    # this rank's rows of the obstacle mask, as the reference holds it: one int per cell
    pin_obst = host_array((nrows, NX), np.int32)
    pin_obst.array[...] = channel_mask(NX, ny, rows=(row0, row0 + nrows))

    lat = make_lattice(ny, row0, nrows, pin_obst.array)
    for _ in range(W):
        lat.run_timed(T)
    mass0 = sum_over_ranks(lat.digest()[0])
    steps0 = lat.info().steps_done
    launches0 = lat.info().kernel_launches
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last_sums = np.empty(T) if args.dump_outputs else None
    dev_ms, wall_s = timed_runs(lat, K, 0, last_sums)
    clocks = sampler.stop() if rank == 0 else None
    launches = lat.info().kernel_launches - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, lat, R, last_sums, ny, row0, nrows)
    mass1 = sum_over_ranks(lat.digest()[0])
    av_tail = lat.run_sums(2)               # sanity: the numbers are finite and positive
    assert np.all(np.isfinite(av_tail)) and np.all(av_tail > 0), av_tail
    info = lat.info()
    lat.close()
    # total mass of the WHOLE lattice over the timed timesteps: collisions and streaming conserve
    # it, accelerate_flow moves it between speeds (d2q9-bgk.c:246-258) -- only float rounding drifts
    parity["mass_conservation_full_grid"] = {
        "timesteps": int(info.steps_done - steps0 - 2), "total_density_before": mass0, "total_density_after": mass1,
        "relative_drift": abs(mass1 - mass0) / mass0, "ok": bool(abs(mass1 - mass0) / mass0 < 1e-4)}
    if parity.get("checked"):
        parity["ok"] = bool(parity["ok"] and parity["mass_conservation_full_grid"]["ok"])

    value = cells_total * T * K / (dev_ms * 1e-3) / 1e6
    two_step = int(info.kernel) == L.KERNEL_TB2
    steps_per_launch = 2 if two_step else 1
    kernel_ms = dev_ms / (T * K) * steps_per_launch               # one launch per pass per GPU
    cells_per_launch = float(NX) * nrows
    # algorithmic bytes: each of the 9 distributions of a cell read once and written once per
    # launch -- 72 B per cell per launch; the two-step kernel advances two timesteps with them
    achieved = cells_per_launch * BYTES_PER_UPDATE / (kernel_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak()
    traffic = ncu_traffic(int(info.kernel))

    # ---- strong scaling of the single 16384-row grid (BASELINE.json configs[3]) --------------
    strong = None
    if not args.no_strong and args.scaling == "weak":
        if world == 1:
            strong = {"value": value, "unit": "MLUPS", "ms_per_timestep": dev_ms / (T * K), "rows_per_gpu": ROWS_PER_GPU,
                      "note": "N = 1: the same grid as `value`"}
        else:
            sny = ROWS_PER_GPU
            srow0, snrows = L.split_rows(sny, world)[rank]
            sobst = L.pack_obstacle_bits(channel_mask(NX, sny, rows=(srow0, srow0 + snrows)))
            slat = make_lattice(sny, srow0, snrows, sobst, bits=True)
            sms, _ = timed_runs(slat, 2, 1)
            sinfo = slat.info()
            slat.close()
            strong = {"value": float(NX) * sny * T * 2 / (sms * 1e-3) / 1e6, "unit": "MLUPS",
                      "ms_per_timestep": sms / (2 * T), "rows_per_gpu": snrows, "timesteps": 2 * T,
                      "kernel": KERNEL_NAMES.get(int(sinfo.kernel), str(sinfo.kernel)),
                      "workload": "the single %dx%d grid split over %d GPUs, device-timed, max over ranks" % (NX, sny, world)}

    # ---- e2e: host buffers -> C-ABI -> host buffers, every step -----------------------
    e2e = None
    if not args.no_e2e:
        out = [host_array((nrows, NX), np.float32) for _ in range(4)]
        av_host = np.empty(T, dtype=np.float32)
        verbose = bool(os.environ.get("LBM_BENCH_VERBOSE"))

        def one_e2e_step(obstacles, bits):
            t = [time.perf_counter()]
            lt = make_lattice(ny, row0, nrows, obstacles, bits=bits); t.append(time.perf_counter())
            lt.run(T, out=av_host); t.append(time.perf_counter())
            lt.final_fields(out=[o.array for o in out]); t.append(time.perf_counter())
            lt.close(); t.append(time.perf_counter())
            if verbose:
                sys.stderr.write("rank %d e2e step: create %.1f run %.1f fields %.1f destroy %.1f ms\n"
                                 % ((rank,) + tuple(1e3 * (b - a) for a, b in zip(t, t[1:]))))

        def e2e_leg(obstacles, bits):
            one_e2e_step(obstacles, bits)        # warm-up (first touch of the pinned pages etc.)
            barrier()
            t0 = time.perf_counter()
            for _ in range(K):
                one_e2e_step(obstacles, bits)
            barrier()
            secs = max_over_ranks(time.perf_counter() - t0)
            assert np.all(np.isfinite(av_host)) and np.isfinite(out[3].array[::997, ::997]).all()
            return secs

        e2e_s = e2e_leg(pin_obst.array, False)
        e2e = {"value": cells_total * T * K / e2e_s / 1e6, "unit": "MLUPS",
               "h2d_bytes_per_step": int(pin_obst.array.nbytes) * world,
               "d2h_bytes_per_step": int(4 * out[0].array.nbytes + av_host.nbytes) * world,
               "ms_per_step": 1e3 * e2e_s / K, "host_memory": host_memory,
               "what": "lbm_gpu_create(LBM_GPU_POOL, int32 obstacles from pinned host) + lbm_gpu_run(T) -> av_vels on host + "
                       "lbm_gpu_final_fields(u_x,u_y,|u|,pressure) -> pinned host + lbm_gpu_destroy"}
        # the same with the obstacle array in the library's packed-bit input format
        # (LBM_GPU_OBST_BITS, include/lbm_gpu.h): 32x fewer bytes to the device
        pin_bits = host_array((nrows, (NX + 31) // 32), np.uint32)
        pin_bits.array[...] = L.pack_obstacle_bits(pin_obst.array)
        bits_s = e2e_leg(pin_bits.array, True)
        e2e["with_bit_packed_mask"] = {"value": cells_total * T * K / bits_s / 1e6, "ms_per_step": 1e3 * bits_s / K,
                                       "h2d_bytes_per_step": int(pin_bits.array.nbytes) * world}
        pin_bits.free()
        for o in out:
            o.free()
    pin_obst.free()

    shipped = None
    if rank == 0 and world == 1 and not args.no_shipped:
        shipped = shipped_block(L)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _, _ = cpu_reference_mlups(12.0)
        serial, _, _ = cpu_reference_mlups(8.0, threads=1, prefer="serial")
        cpu["serial_value"] = serial["value"]
        cpu["serial_sample"] = serial["sample"]

    R.close()
    if rank != 0:
        return 0 if parity.get("ok", True) else 1

    bytes_per_update = BYTES_PER_UPDATE / steps_per_launch
    line = {
        "metric": "MLUPS (d2q9-bgk lattice updates per second / 1e6)",
        "value": value, "unit": "MLUPS", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, world), cpu_binding=binding),
        "achieved_hbm_gbs_per_gpu": achieved,
        "wall_ms_per_step": 1e3 * wall_s / K,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic["dram_bytes_per_launch"],
                     "traffic_source": traffic["source"], "library_sha256_16": library_id(L),
                     "peak_source": peak_src,
                     "frac_of_8tbs_datasheet": achieved / 8000.0,   # frac > 1 means: faster than a plain copy
                     "algorithmic_bytes_per_launch": cells_per_launch * BYTES_PER_UPDATE,
                     "timesteps_per_launch": steps_per_launch,
                     "algorithmic_bytes_per_update": bytes_per_update,
                     "equivalent_72B_per_update": {
                         "gbs": value / world * BYTES_PER_UPDATE * 1e-3, "frac": value / world * BYTES_PER_UPDATE * 1e-3 / peak,
                         "note": "what a one-timestep-per-pass kernel (72 B per update) would need for the same MLUPS"},
                     "kernel": KERNEL_NAMES.get(int(info.kernel), str(info.kernel)), "kernel_ms": kernel_ms},
        "cpu_baseline": cpu,
        "e2e": e2e,
        "parity": parity,
        "strong": strong,
        "shipped": shipped,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "kernel_variant": int(info.kernel),
    }
    print(json.dumps(line), flush=True)
    return 0 if parity.get("ok", True) else 1


if __name__ == "__main__":
    sys.exit(main())
