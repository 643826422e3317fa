"""lbm_gpu_obstacle_force against tests/force_ref.py bit for bit: every kernel family and precision,
1-3 slabs on one GPU, ragged widths, obstacles on the wrap edges, slab edges and rows ny-2 / ny-1,
overlapping, empty and edge-touching boxes, and a grid of many blocks.  Also the momentum balance
per step, run(a); force; run(b) == run(a + b), NaN confined to its boxes, refusals that leave the
handle unchanged, the shares of slab handles across processes, and the CLI's forces.dat."""
import ctypes as C
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import force_ref as F
import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "d2q9-bgk")
F16 = L.STORE_F16


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def inputs(nx, ny, seed=5, p_obst=0.06):
    """A random lattice whose mask also has obstacles on both wrap edges, on rows 0, ny-2, ny-1, and
    on the rows next to every cut of a 2- or 3-slab split."""
    cells, obst = O.random_lattice(nx, ny, seed=seed, p_obst=p_obst)
    rng = np.random.default_rng(seed)
    rows = {ny - 1, ny - 2}
    for n in (2, 3):
        for r0, k in L.split_rows(ny, n):
            rows |= {r0, (r0 - 1) % ny, (r0 + k - 1) % ny}
    for r in rows:
        obst[r] |= (rng.random(nx) < 0.3).astype(np.int32)
    return cells, obst


def boxes_for(nx, ny):
    """overlapping, empty, edge-touching, single-row and single-column boxes, and the whole grid"""
    return np.array([(0, 0, nx, ny), (0, 0, nx // 2, ny // 2), (nx // 3, ny // 4, nx, ny), (0, 0, 0, 0),
                     (nx - 1, 0, nx, ny), (0, ny - 2, nx, ny - 1), (0, ny - 1, nx, ny), (5, 3, 5, ny),
                     (1, 1, nx - 1, ny - 1), (0, 0, nx, 1)], dtype=np.int32)


def expected(lat, obst, boxes, density=D):
    cells = lat.download()                                  # decoded fp32 for binary16
    return F.force(F.accelerated(cells, obst, density, A), obst, boxes)


def make(nx, ny, cells, obst, flags=0, f64=False, n_gpus=1):
    if f64:
        cells = cells.astype(np.float64)
    return L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=flags, f64=f64, n_gpus=n_gpus,
                     device_ids=[0] * n_gpus)


# (id, nx, ny, flags, f64, kernel the handle must run)
FAMILIES = [
    ("K1a", 256, 96, L.KERNEL_VEC4, False, L.KERNEL_VEC4),
    ("K1b", 130, 64, L.KERNEL_SCALAR, False, L.KERNEL_SCALAR),
    ("K1c", 1100, 40, L.KERNEL_TMA, False, L.KERNEL_TMA),
    ("K5", 512, 512, 0, False, L.KERNEL_PERSISTENT),
    ("K6", 128, 128, L.KERNEL_CLUSTER, False, L.KERNEL_CLUSTER),
    ("K7", 512, 64, L.KERNEL_TB2, False, L.KERNEL_TB2),
    ("K9", 128, 128, 0, False, L.KERNEL_PAIRS),
    ("K10", 256, 64, L.KERNEL_TB3, False, L.KERNEL_TB3),
    ("f64-K1a", 256, 96, L.KERNEL_VEC4, True, L.KERNEL_VEC4),
    ("f64-K5", 128, 128, 0, True, L.KERNEL_PERSISTENT),
    ("K1a-f16", 68, 32, F16, False, L.KERNEL_VEC4),
    ("K7-f16", 64, 32, F16, False, L.KERNEL_TB2),
]


@pytest.mark.parametrize("strict", [0, L.STRICT], ids=["default", "strict"])
@pytest.mark.parametrize("fam", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_every_kernel_family_matches_the_restatement(fam, strict):
    _, nx, ny, flags, f64, kernel = fam
    cells, obst = inputs(nx, ny)
    boxes = boxes_for(nx, ny)
    with make(nx, ny, cells, obst, flags | strict, f64) as lat:
        assert lat.info().kernel == kernel
        for steps in (0, 5, 2, 1):                          # odd tails of K7, K9 and K10 included
            lat.run(steps)
            got = lat.obstacle_force(boxes)
            want = expected(lat, obst, boxes)
            assert np.array_equal(bits(got), bits(want)), (steps, got, want)
            assert np.array_equal(bits(lat.obstacle_force()), bits(want[:1]))


@pytest.mark.parametrize("f64", [False, True], ids=["f32", "f64"])
@pytest.mark.parametrize("nx", [128, 37, 133])
def test_slab_splits_give_the_bits_of_one_slab(nx, f64):
    ny = 45
    cells, obst = inputs(nx, ny, seed=nx)
    boxes = boxes_for(nx, ny)
    results = []
    for n in (1, 2, 3):
        with make(nx, ny, cells, obst, L.KERNEL_VEC4 if nx % 4 else 0, f64, n_gpus=n) as lat:
            lat.run(7)
            results.append(lat.obstacle_force(boxes))
            if n == 1:
                want = expected(lat, obst, boxes)
    for got in results:
        assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("n", [2, 3])
def test_multi_slab_two_step_kernel(n):
    """K7 on several slabs pushes deep ghost rows; the force reads depth 0 after every pass length."""
    nx, ny = 128, 45
    cells, obst = inputs(nx, ny, seed=8)
    boxes = boxes_for(nx, ny)
    with make(nx, ny, cells, obst, L.KERNEL_TB2, n_gpus=n) as lat, make(nx, ny, cells, obst, L.KERNEL_TB2) as one:
        assert lat.info().kernel == L.KERNEL_TB2 and lat.info().n_gpus == n
        for steps in (4, 1, 2, 3):
            lat.run(steps)
            one.run(steps)
            want = expected(lat, obst, boxes)
            assert np.array_equal(bits(lat.obstacle_force(boxes)), bits(want))
            assert np.array_equal(bits(one.obstacle_force(boxes)), bits(want))


@pytest.mark.parametrize("n_gpus", [1, 3])
def test_256_small_boxes(n_gpus):
    """the most boxes a call takes: random sizes and places, many across the slab cuts, some empty"""
    nx, ny = 520, 300
    cells, obst = inputs(nx, ny, seed=12, p_obst=0.03)
    rng = np.random.default_rng(12)
    x0 = rng.integers(0, nx, 256)
    y0 = rng.integers(0, ny, 256)
    boxes = np.stack([x0, y0, np.minimum(x0 + rng.integers(0, 70, 256), nx),
                      np.minimum(y0 + rng.integers(0, 70, 256), ny)], axis=1).astype(np.int32)
    boxes[0] = (0, 0, nx, ny)
    with make(nx, ny, cells, obst, L.KERNEL_VEC4, n_gpus=n_gpus) as lat:
        lat.run(3)
        assert np.array_equal(bits(lat.obstacle_force(boxes)), bits(expected(lat, obst, boxes)))


def test_many_blocks():
    nx, ny = 8190, 2600
    cells, obst = O.random_lattice(nx, 64, seed=9, p_obst=0.01)
    cells = np.tile(cells, (-(-ny // 64), 1, 1))[:ny]
    obst = np.tile(obst, (-(-ny // 64), 1))[:ny]
    obst[ny - 3:] |= (np.random.default_rng(9).random((3, nx)) < 0.2).astype(np.int32)
    boxes = np.array([(0, 0, nx, ny), (100, 50, 4100, 2000), (4000, 0, nx, ny)], dtype=np.int32)
    with make(nx, ny, cells, obst, n_gpus=1) as lat:
        lat.run(3)
        assert np.array_equal(bits(lat.obstacle_force(boxes)), bits(expected(lat, obst, boxes)))


def test_batch_members():
    nx, ny, n = 128, 64, 3
    lats = []
    try:
        for i in range(n):
            cells, obst = inputs(nx, ny, seed=30 + i)
            lats.append((L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst), obst))
        L.run_batch([l for l, _ in lats], 5)
        for lat, obst in lats:
            assert np.array_equal(bits(lat.obstacle_force(boxes_for(nx, ny))), bits(expected(lat, obst, boxes_for(nx, ny))))
    finally:
        for lat, _ in lats:
            lat.close()


@pytest.mark.parametrize("strict", [0, L.STRICT], ids=["default", "strict"])
def test_momentum_balance_per_step(strict):
    """P_fluid(t+1) = P~_fluid(t) - F_all(t) within the bound of tests/test_force_ref.py."""
    nx, ny = 256, 128
    cells, obst = inputs(nx, ny, seed=17)
    with make(nx, ny, cells, obst, strict) as lat:
        for _ in range(4):
            f_all = lat.obstacle_force()[0]
            state = lat.download()
            p_tilde = np.array(F.fluid_momentum(F.accelerated(state, obst, D, A), obst))
            lat.run(1)
            new = lat.download()
            p_new = np.array(F.fluid_momentum(new, obst))
            bound = (3 * np.finfo(np.float32).eps * float(np.abs(new).max()) * int((obst == 0).sum())
                     + 16 * 2.0 ** -33 * int(obst.sum()))
            err = np.abs(p_new - (p_tilde - f_all))
            assert (err <= bound).all(), (err, bound)
            assert err.max() < 1e-3 * np.abs(f_all).max()       # the force is far above the rounding


@pytest.mark.parametrize("flags", [0, L.KERNEL_TB3, F16], ids=["K9", "K10", "f16"])
def test_force_between_runs_changes_nothing(flags):
    nx, ny = (256, 64) if flags else (128, 128)
    cells, obst = inputs(nx, ny, seed=2)
    with make(nx, ny, cells, obst, flags) as ref:
        av_ref = ref.run(12)
        dig_ref = ref.digest()
        info_ref = ref.info()
    with make(nx, ny, cells, obst, flags) as lat:
        av_a = lat.run(5)
        lat.obstacle_force(boxes_for(nx, ny))
        assert lat.info().steps_done == 5 and lat.info().kernel == info_ref.kernel
        av_b = lat.run(7)
        assert lat.digest() == dig_ref and lat.info().steps_done == 12
    assert np.array_equal(np.concatenate([av_a, av_b]).view(np.uint32), av_ref.view(np.uint32))


def test_nan_stays_in_its_boxes():
    nx, ny = 64, 32
    cells, obst = inputs(nx, ny, seed=4)
    obst[10, 10] = 1
    obst[10, 11] = 0
    cells[10, 10, 1] = np.nan                              # leaves the solid cell towards (11, 10)
    boxes = np.array([(0, 0, nx, ny), (8, 8, 12, 12), (20, 0, nx, ny), (0, 20, nx, ny)], dtype=np.int32)
    with make(nx, ny, cells, obst, L.KERNEL_VEC4) as lat:
        got = lat.obstacle_force(boxes)
        want = expected(lat, obst, boxes)
    assert np.isnan(got[:2]).all() and np.isfinite(got[2:]).all()
    assert np.array_equal(bits(got[2:]), bits(want[2:]))


def test_refusals_leave_the_handle_unchanged():
    nx, ny = 64, 32
    cells, obst = inputs(nx, ny, seed=6)
    lib = L.load_library()
    with make(nx, ny, cells, obst) as lat:
        lat.run(3)
        before = lat.digest(), lat.info().steps_done, lat.info().kernel_launches
        good = lat.obstacle_force()
        launches = lat.info().kernel_launches
        out = np.full((300, 2), 7.0)
        box = np.array([[0, 0, nx, ny]] * 300, dtype=np.int32)

        def refused(n, b, o, why):
            rc = lib.lbm_gpu_obstacle_force(lat.h, n, None if b is None else b.ctypes.data_as(C.c_void_p),
                                            None if o is None else o.ctypes.data_as(C.c_void_p))
            msg = lib.lbm_gpu_last_error().decode()
            assert rc != 0 and msg.startswith("lbm_gpu_obstacle_force:") and why in msg, msg
        refused(0, box, out, "n_boxes 0")
        refused(257, box, out, "n_boxes 257")
        refused(1, box, None, "NULL force_out")
        refused(2, None, out, "boxes is NULL")
        for j, bad in enumerate([(-1, 0, 1, 1), (0, 0, nx + 1, 1), (3, 0, 2, 1), (0, 5, 1, 4), (0, 0, 1, ny + 1)]):
            b = box[:4].copy()
            b[2] = bad
            refused(4, b, out, "box 2 ")
        assert (out == 7.0).all()
        assert lat.info().kernel_launches == launches
        assert (lat.digest(), lat.info().steps_done) == before[:2]
        assert np.array_equal(bits(lat.obstacle_force()), bits(good))


def test_slab_handle_refusals_in_one_process():
    """A slab handle that holds part of the grid is refused until it is connected, and again after
    lbm_gpu_load_rows until lbm_gpu_ipc_prepare: its ghost rows would be stale."""
    nx, ny = 64, 32
    cells, obst = inputs(nx, ny, seed=13)
    with L.Lattice(nx, ny, D, A, W, cells=cells[:16], obstacles=obst[:16], slab=(0, 16), device_ids=[0]) as lat:
        with pytest.raises(L.LbmError, match="^lbm_gpu_obstacle_force: lattice is not connected"):
            lat.obstacle_force()
        lat.load_rows(0, lat.save_rows())
        with pytest.raises(L.LbmError, match="^lbm_gpu_obstacle_force: rows were loaded .*lbm_gpu_ipc_prepare"):
            lat.obstacle_force()


# ------------------------------------------------------------------ multi-GPU, one process per GPU
WORKER = textwrap.dedent("""
    import os, sys
    import numpy as np
    sys.path.insert(0, %(root)r); sys.path.insert(0, os.path.join(%(root)r, "tests"))
    import torch, torch.distributed as dist
    import lbm_b200 as L
    import oracle_lib as O
    from importlib import import_module
    slabs = import_module("advanced-hpc-lbm_b200.slabs")
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nx, ny, out = %(nx)d, %(ny)d, %(out)r
    cells, obst = O.random_lattice(nx, ny, seed=21, p_obst=0.05)
    boxes = np.array(%(boxes)r, dtype=np.int32)
    r0, k = L.split_rows(ny, world)[rank]
    lat = L.Lattice(nx, ny, 0.1, 0.005, 1.85, cells=cells[r0:r0 + k], obstacles=obst[r0:r0 + k], slab=(r0, k),
                    device_ids=[local])
    lat.ipc_connect_all(slabs.gather_descriptors(lat.ipc_export(), world, dist))
    dist.barrier(); lat.ipc_prepare(); dist.barrier()
    lat.run_sums(5)
    np.save(os.path.join(out, "share_%%d.npy" %% rank), lat.obstacle_force(boxes))
    np.save(os.path.join(out, "rows_%%d.npy" %% rank), lat.save_rows())
    lat.load_rows(r0, lat.save_rows())
    try:
        lat.obstacle_force(boxes)
        msg = "no error"
    except L.LbmError as e:
        msg = str(e)
    open(os.path.join(out, "refused_%%d.txt" %% rank), "w").write(msg)
    dist.barrier(); lat.ipc_prepare(); dist.barrier()
    np.save(os.path.join(out, "again_%%d.npy" %% rank), lat.obstacle_force(boxes))
    lat.close()
    dist.barrier()
    dist.destroy_process_group()
""")


def test_slab_shares_add_up_across_processes(tmp_path):
    n = min(L.load_library().lbm_gpu_device_count(), 4)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    nx, ny = 256, 203
    boxes = [(0, 0, nx, ny), (10, 40, 200, 150), (0, 100, nx, 103)]
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT, "nx": nx, "ny": ny, "out": str(tmp_path), "boxes": boxes})
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=%d" % n,
                        "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-4000:]
    cells, obst = O.random_lattice(nx, ny, seed=21, p_obst=0.05)
    with make(nx, ny, cells, obst) as one:
        one.run(5)
        whole = one.obstacle_force(np.array(boxes, dtype=np.int32))
    rec = np.concatenate([np.load(str(tmp_path / ("rows_%d.npy" % i))) for i in range(n)])
    tilde = F.accelerated(rec, obst, D, A)
    total = np.zeros_like(whole)
    for i, (r0, k) in enumerate(L.split_rows(ny, n)):
        share = np.load(str(tmp_path / ("share_%d.npy" % i)))
        assert np.array_equal(bits(share), bits(F.force(tilde, obst, boxes, rows=(r0, r0 + k))))
        assert np.array_equal(bits(np.load(str(tmp_path / ("again_%d.npy" % i)))), bits(share))
        msg = (tmp_path / ("refused_%d.txt" % i)).read_text()
        assert msg.startswith("lbm_gpu_obstacle_force:") and "lbm_gpu_ipc_prepare" in msg, msg
        total += share
    assert np.allclose(total, whole, rtol=n * 2.0 ** -52, atol=0)


# ------------------------------------------------------------------------------------------- CLI
def cli(cwd, params, env_extra):
    env = dict(os.environ)
    for k in ("LBM_CHECKPOINT", "LBM_CHECKPOINT_EVERY", "LBM_RESTART", "LBM_FORCE_EVERY", "LBM_FORCE_BOXES"):
        env.pop(k, None)
    env.update(env_extra)
    r = subprocess.run([EXE, params, os.path.join(ROOT, "inputs", "obstacles_128x128.dat")], cwd=str(cwd), env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    return r


def test_cli_forces_dat(tmp_path):
    lines = open(os.path.join(ROOT, "inputs", "input_128x128.params")).read().split("\n")
    nx, ny, density, accel, omega = int(lines[0]), int(lines[1]), float(lines[4]), float(lines[5]), float(lines[6])
    lines[2] = "700"
    full = tmp_path / "full.params"
    full.write_text("\n".join(lines))
    lines[2] = "300"
    short = tmp_path / "short.params"
    short.write_text("\n".join(lines))
    spec = "0,0,128,128;20,1,60,127;0,0,128,1"
    boxes = np.array([[int(v) for v in b.split(",")] for b in spec.split(";")], dtype=np.int32)
    plain, knob, part = tmp_path / "plain", tmp_path / "knob", tmp_path / "part"
    for d in (plain, knob, part):
        d.mkdir()
    cli(plain, str(full), {})
    cli(knob, str(full), {"LBM_FORCE_EVERY": "120", "LBM_FORCE_BOXES": spec})
    for name in ("av_vels.dat", "final_state.dat"):
        assert (knob / name).read_bytes() == (plain / name).read_bytes()
    got = (knob / "forces.dat").read_text().splitlines()
    assert len(got) == 5                                    # t = 120, 240, ..., 600 <= 700
    obst = np.zeros((ny, nx), dtype=np.int32)
    for line in open(os.path.join(ROOT, "inputs", "obstacles_128x128.dat")):
        if line.strip():
            x, y, _ = map(int, line.split())
            obst[y, x] = 1
    with L.Lattice(nx, ny, density, accel, omega, obstacles=obst) as lat:
        want = []
        for t in range(120, 701, 120):
            lat.run(120)
            f = lat.obstacle_force(boxes)
            want.append("\t".join(["%d" % t] + ["%.12E" % v for v in f.ravel()]))
    assert got == want
    # restart: only the samples after the restart step, equal to the uninterrupted run's lines
    ckpt = tmp_path / "run.ckpt"
    cli(part, str(short), {"LBM_CHECKPOINT": str(ckpt)})
    cli(part, str(full), {"LBM_RESTART": str(ckpt), "LBM_FORCE_EVERY": "120", "LBM_FORCE_BOXES": spec})
    assert (part / "forces.dat").read_text().splitlines() == got[2:]
    for name in ("av_vels.dat", "final_state.dat"):
        assert (part / name).read_bytes() == (plain / name).read_bytes()
