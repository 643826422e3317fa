"""Checkpoint and restart (lbm_gpu_save_rows / lbm_gpu_load_rows, LBM_CHECKPOINT / LBM_RESTART):
run(a); save; [new handle, other slab layout, other process] load; run(b) must give the bits of
run(a + b) -- lattice records, av_vels (as uint32 / uint64) and the digest checksum -- for every
kernel family, and the CLI's outputs must equal an uninterrupted run's byte for byte."""
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "d2q9-bgk")
F16 = L.STORE_F16


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view({2: np.uint16, 4: np.uint32, 8: np.uint64}[a.dtype.itemsize])


def lattice_inputs(nx, ny, seed=7):
    if nx * ny <= (1 << 22):
        return O.random_lattice(nx, ny, seed=seed, p_obst=0.03)
    # large grids: a random band of 64 rows repeated (generating every row costs minutes of host time)
    cells, obst = O.random_lattice(nx, 64, seed=seed, p_obst=0.03)
    reps = -(-ny // 64)
    return np.tile(cells, (reps, 1, 1))[:ny], np.tile(obst, (reps, 1))[:ny]


def make(nx, ny, cells, obst, flags=0, f64=False, n_gpus=1, device_ids=None, density=D):
    if f64 and cells is not None:
        cells = cells.astype(np.float64)
    return L.Lattice(nx, ny, density, A, W, cells=cells, obstacles=obst, flags=flags, f64=f64, n_gpus=n_gpus,
                     device_ids=device_ids)


# (id, nx, ny, flags, f64, kernel the handle must run)
FAMILIES = [
    ("K9", 128, 128, 0, False, L.KERNEL_PAIRS),
    ("K5", 512, 512, 0, False, L.KERNEL_PERSISTENT),
    ("K1a", 256, 96, L.KERNEL_VEC4, False, L.KERNEL_VEC4),
    ("K1b", 130, 64, L.KERNEL_SCALAR, False, L.KERNEL_SCALAR),
    ("K1c", 1100, 40, L.KERNEL_TMA, False, L.KERNEL_TMA),
    ("K7", 512, 64, L.KERNEL_TB2, False, L.KERNEL_TB2),
    ("K10", 16384, 2048, 0, False, L.KERNEL_TB3),
    ("f64-K1a", 256, 96, L.KERNEL_VEC4, True, L.KERNEL_VEC4),
    ("f64-K5", 128, 128, 0, True, L.KERNEL_PERSISTENT),
    ("K1a-f16", 68, 32, F16, False, L.KERNEL_VEC4),
    ("K7-f16", 64, 32, F16, False, L.KERNEL_TB2),
]


@pytest.mark.parametrize("strict", [0, L.STRICT], ids=["default", "strict"])
@pytest.mark.parametrize("ab", [(1, 6), (2, 7), (5, 4)], ids=lambda ab: "%d+%d" % ab)
@pytest.mark.parametrize("fam", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_restart_in_a_fresh_handle_equals_one_run(fam, ab, strict):
    """a < 3 puts the odd tails (K1a after K7, K7 or K1a after K10, K1a after K9) across the restart."""
    _, nx, ny, flags, f64, kernel = fam
    a, b = ab
    cells, obst = lattice_inputs(nx, ny)
    with make(nx, ny, cells, obst, flags | strict, f64) as ref:
        assert ref.info().kernel == kernel
        av_ref = ref.run(a + b)
        dig_ref = ref.digest()
        rec_ref = ref.save_rows(0, 8), ref.save_rows(ny - 3, 3)
    with make(nx, ny, cells, obst, flags | strict, f64) as first:
        av_a = first.run(a)
        rec = first.save_rows()
        assert rec.dtype == first.record_dtype and rec.shape == (ny, nx, 9)
    with make(nx, ny, None, obst, flags | strict, f64) as second:      # rest state, replaced by the load
        second.load_rows(0, rec)
        del rec
        assert second.info().steps_done == 0 and second.info().kernel == kernel
        av_b = second.run(b)
        assert second.digest()[1] == dig_ref[1]
        assert np.array_equal(bits(second.save_rows(0, 8)), bits(rec_ref[0]))
        assert np.array_equal(bits(second.save_rows(ny - 3, 3)), bits(rec_ref[1]))
    assert np.array_equal(bits(np.concatenate([av_a, av_b])), bits(av_ref))


@pytest.mark.parametrize("src,dst", [(1, 3), (3, 1)])
def test_restart_into_another_slab_layout(src, dst):
    nx, ny, a, b = 128, 64, 5, 8
    cells, obst = lattice_inputs(nx, ny, seed=3)
    with make(nx, ny, cells, obst) as ref:
        av_ref = ref.run(a + b)
        rec_ref = ref.save_rows()
        dig_ref = ref.digest()
    with make(nx, ny, cells, obst, n_gpus=src, device_ids=[0] * src) as first:
        av_a = first.run(a)
        rec = first.save_rows()
    with make(nx, ny, None, obst, n_gpus=dst, device_ids=[0] * dst) as second:
        second.load_rows(0, rec)
        av_b = second.run(b)
        assert np.array_equal(bits(second.save_rows()), bits(rec_ref))
        assert second.digest() == dig_ref
    assert np.array_equal(bits(np.concatenate([av_a, av_b])), bits(av_ref))


def chunks(ny, rng):
    """Row chunks covering [0, ny) in random order: single rows, the last three rows on their own."""
    cuts = sorted(set([0, 1, 2, ny - 3, ny - 2, ny - 1, ny] + list(rng.integers(1, ny, size=8))))
    out = [(r0, r1 - r0) for r0, r1 in zip(cuts[:-1], cuts[1:])]
    rng.shuffle(out)
    return out


@pytest.mark.parametrize("n_slabs", [1, 3])
@pytest.mark.parametrize("nx,flags", [(128, 0), (37, 0), (133, L.KERNEL_VEC4), (68, F16), (64, F16)])
def test_loads_in_any_row_chunks(nx, flags, n_slabs):
    """Chunks of any size in any order, across slab boundaries, including rows 0, ny-2 and ny-1;
    ragged widths (nx not a multiple of 4 or 32) keep their padding columns out of it."""
    if flags & F16 and n_slabs > 1:
        pytest.skip("binary16 lattices are single-slab")
    ny, a, b = 41, 4, 7
    rng = np.random.default_rng(nx + n_slabs)
    cells, obst = lattice_inputs(nx, ny, seed=5)
    with make(nx, ny, cells, obst, flags) as ref:
        av_ref = ref.run(a + b)
        rec_ref = ref.save_rows()
    with make(nx, ny, cells, obst, flags) as first:
        av_a = first.run(a)
        rec = first.save_rows()
    with make(nx, ny, None, obst, flags, n_gpus=n_slabs, device_ids=[0] * n_slabs) as second:
        for r0, n in chunks(ny, rng):
            second.load_rows(r0, rec[r0:r0 + n])
        assert np.array_equal(bits(second.save_rows()), bits(rec))
        for r0, n in chunks(ny, rng):
            assert np.array_equal(bits(second.save_rows(r0, n)), bits(rec[r0:r0 + n]))
        av_b = second.run(b)
        assert np.array_equal(bits(second.save_rows()), bits(rec_ref))
    assert np.array_equal(bits(np.concatenate([av_a, av_b])), bits(av_ref))


@pytest.mark.parametrize("f64", [False, True])
def test_several_staging_chunks_per_call(f64):
    """4096 x 1024 fp32 is 144 MiB of records (fp64 288 MiB): several 32 MiB staging halves per call."""
    nx, ny = 4096, 1024
    cells, obst = lattice_inputs(nx, ny, seed=11)
    with make(nx, ny, cells, obst, f64=f64) as lat:
        lat.run(3)
        rec = lat.save_rows()
        down = lat.download()
        assert rec.tobytes() == down.tobytes()
        dig = lat.digest()
    with make(nx, ny, None, obst, f64=f64) as other:
        other.load_rows(0, rec)
        assert other.digest() == dig


@pytest.mark.parametrize("nx,ny,n_slabs", [(128, 64, 1), (37, 29, 3), (4096, 300, 2)])
def test_fp32_records_are_download_rows_byte_for_byte(nx, ny, n_slabs):
    cells, obst = lattice_inputs(nx, ny, seed=2)
    with make(nx, ny, cells, obst, n_gpus=n_slabs, device_ids=[0] * n_slabs) as lat:
        lat.run(3)
        for r0, n in [(0, ny), (1, ny - 2), (ny - 2, 2), (ny // 2, 1), (5, 0)]:
            assert lat.save_rows(r0, n).tobytes() == lat.download_rows(r0, n).tobytes()


def test_fp64_records_are_download_f64_byte_for_byte():
    nx, ny = 133, 50
    cells, obst = lattice_inputs(nx, ny, seed=4)
    with make(nx, ny, cells, obst, f64=True, n_gpus=2, device_ids=[0, 0]) as lat:
        lat.run(5)
        assert lat.save_rows().tobytes() == lat.download().tobytes()


def test_f16_round_trip_keeps_the_stored_bits_where_upload_does_not():
    """At density 10 decode-then-encode changes 8195 of the finite binary16 values (numpy, over all
    of them and the three shifts), so upload(download()) moves the stored bits; load_rows(save_rows())
    is the identity on them.  The decoded fp32 values come back the same either way (every changed
    pattern decodes to the value the old one did), so the digest, which reads decoded values, and
    the continued run cannot tell the two apart: only the records show the difference."""
    nx, ny, density = 128, 64, 10.0
    _, obst = O.random_lattice(nx, ny, seed=9, density=density, p_obst=0.03)
    # near the rest state the stored values s_k = f_k - c_k are small, which is where decoding
    # (s_k + c_k, rounded in fp32) drops their low bits
    w = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4, dtype=np.float32) * np.float32(density)
    rng = np.random.default_rng(9)
    cells = (w * (1 + 2e-6 * rng.standard_normal((ny, nx, 9)))).astype(np.float32)
    with L.Lattice(nx, ny, density, A, W, cells=cells, obstacles=obst, flags=F16) as lat, \
            L.Lattice(nx, ny, density, A, W, obstacles=obst, flags=F16) as twin:
        lat.run(2)
        rec = lat.save_rows()
        assert rec.dtype == np.uint16
        dig = lat.digest()
        lat.load_rows(0, rec)
        assert np.array_equal(lat.save_rows(), rec)
        assert lat.digest() == dig
        twin.upload(lat.download())
        moved = twin.save_rows()
        assert np.count_nonzero(moved != rec) > 0
        assert twin.digest() == dig
        lat.run(5)
        twin.run(5)
        assert twin.digest() == lat.digest()
        twin.load_rows(0, rec)                    # the records bring the stored bits back
        assert np.array_equal(twin.save_rows(), rec)


def test_load_between_overlapped_three_step_runs():
    """K10 passes of one run overlap and wait per tile; a load between two K10 runs replaces the
    lattice under the next run's first pass, which waits for the whole previous grid."""
    nx, ny, a, b = 16384, 2048, 6, 9
    cells, obst = lattice_inputs(nx, ny, seed=13)
    with make(nx, ny, cells, obst) as ref:
        assert ref.info().kernel == L.KERNEL_TB3
        av_ref = ref.run(a + b)
        dig_ref = ref.digest()
    with make(nx, ny, cells, obst) as src:
        av_a = src.run(a)
        rec = src.save_rows()
    other, _ = lattice_inputs(nx, ny, seed=14)
    with make(nx, ny, other, obst) as lat:
        lat.run(9)                                # K10 passes, then a load straight after them
        lat.load_rows(0, rec)
        av_b = lat.run(b)
        assert lat.digest()[1] == dig_ref[1]
    assert np.array_equal(bits(np.concatenate([av_a, av_b])), bits(av_ref))


def test_refusals_leave_every_handle_unchanged():
    nx, ny = 64, 20
    cells, obst = lattice_inputs(nx, ny, seed=1)
    lib = L.load_library()
    buf = np.zeros((ny, nx, 9), dtype=np.float32)
    with make(nx, ny, cells, obst) as lat, make(nx, ny, cells, obst, n_gpus=2, device_ids=[0, 0]) as two:
        lat.run(3)
        two.run(3)
        before = [(h.digest(), h.info().steps_done) for h in (lat, two)]
        for h in (lat, two):
            for call, args, msg in [
                (lib.lbm_gpu_load_rows, (0, 1, None), "NULL input"),
                (lib.lbm_gpu_save_rows, (0, 1, None), "NULL output"),
                (lib.lbm_gpu_load_rows, (0, -1, buf.ctypes.data), "negative nrows"),
                (lib.lbm_gpu_save_rows, (0, -1, buf.ctypes.data), "negative nrows"),
                (lib.lbm_gpu_load_rows, (ny - 2, 3, buf.ctypes.data), "not held by this process"),
                (lib.lbm_gpu_load_rows, (-1, 2, buf.ctypes.data), "not held by this process"),
                (lib.lbm_gpu_save_rows, (ny, 1, buf.ctypes.data), "not held by this process"),
            ]:
                assert call(h.h, *args) != 0
                err = lib.lbm_gpu_last_error().decode()
                assert msg in err and err.startswith(call.__name__), err
            assert lib.lbm_gpu_load_rows(h.h, 3, 0, None) == 0     # nrows = 0: nothing to do
            assert lib.lbm_gpu_save_rows(h.h, 3, 0, None) == 0
        with pytest.raises(L.LbmError, match="records of this lattice are float32"):
            lat.load_rows(0, np.zeros((1, nx, 9), dtype=np.float64))
        with pytest.raises(L.LbmError, match="need shape"):
            lat.load_rows(0, np.zeros((1, nx + 1, 9), dtype=np.float32))
        assert [(h.digest(), h.info().steps_done) for h in (lat, two)] == before


def test_slab_handle_saves_and_loads_only_its_rows():
    """A slab handle holding part of the grid serves its own rows; unconnected, it cannot run
    (on one GPU two such handles cannot be connected, so the refusal after a load that waits
    for lbm_gpu_ipc_prepare is checked in the multi-GPU test)."""
    nx, ny = 64, 30
    cells, obst = lattice_inputs(nx, ny, seed=6)
    with L.Lattice(nx, ny, D, A, W, cells=cells[10:20], obstacles=obst[10:20], slab=(10, 10)) as s:
        rec = s.save_rows()
        assert rec.shape == (10, nx, 9) and np.array_equal(rec, cells[10:20])
        with pytest.raises(L.LbmError, match="lbm_gpu_save_rows: row range is not held"):
            s.save_rows(9, 2)
        s.load_rows(12, cells[12:15] * 2)
        assert np.array_equal(s.save_rows(12, 3), cells[12:15] * 2)
        with pytest.raises(L.LbmError, match="not connected"):
            s.run(1)


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
    nx, ny, a, b, out, phase = %(nx)d, %(ny)d, %(a)d, %(b)d, %(out)r, %(phase)r
    cells, obst = O.random_lattice(nx, ny, seed=21, p_obst=0.02)
    r0, k = L.split_rows(ny, world)[rank]
    init = cells[r0:r0 + k] if phase == "save" else None
    lat = L.Lattice(nx, ny, 0.1, 0.005, 1.85, cells=init, obstacles=obst[r0:r0 + k], slab=(r0, k), device_ids=[local])
    lat.ipc_connect_all(slabs.gather_descriptors(lat.ipc_export(), world, dist))
    dist.barrier(); lat.ipc_prepare(); dist.barrier()
    if phase == "save":
        sums = lat.run_sums(a)
        np.save(os.path.join(out, "sums_a_%%d.npy" %% rank), sums)
        np.save(os.path.join(out, "rows_%%d.npy" %% rank), lat.save_rows())
    else:
        # the rows of the whole grid, saved by another number of ranks: take this rank's
        rec = np.concatenate([np.load(os.path.join(out, f)) for f in sorted(
            (f for f in os.listdir(out) if f.startswith("rows_")), key=lambda f: int(f[5:-4]))])
        lat.load_rows(r0, rec[r0:r0 + k])
        try:
            lat.run_sums(1)
            msg = "no error"
        except L.LbmError as e:
            msg = str(e)
        open(os.path.join(out, "refused_%%d.txt" %% rank), "w").write(msg)
        dist.barrier(); lat.ipc_prepare(); dist.barrier()
        sums = lat.run_sums(b)
        np.save(os.path.join(out, "sums_b_%%d.npy" %% rank), sums)
        np.save(os.path.join(out, "final_%%d.npy" %% rank), lat.save_rows())
    lat.close()
    dist.barrier()
    dist.destroy_process_group()
""")


def _launch(tmp_path, n, phase, nx, ny, a, b):
    script = tmp_path / ("worker_%s.py" % phase)
    script.write_text(WORKER % {"root": ROOT, "nx": nx, "ny": ny, "a": a, "b": b, "out": str(tmp_path), "phase": phase})
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=%d" % n,
           "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)]
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)


def test_ranks_save_and_restore_into_another_split(tmp_path):
    """n ranks save their rows; n-1 ranks (or one process) load them and continue."""
    n = min(L.load_library().lbm_gpu_device_count(), 4)
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    nx, ny, a, b = 512, 203, 5, 8
    r = _launch(tmp_path, n, "save", nx, ny, a, b)
    assert r.returncode == 0, r.stdout[-4000:]
    cells, obst = O.random_lattice(nx, ny, seed=21, p_obst=0.02)
    with make(nx, ny, cells, obst) as ref:
        ref.run(a + b)
        rec_ref = ref.save_rows()
        dig_ref = ref.digest()
    rec = np.concatenate([np.load(str(tmp_path / ("rows_%d.npy" % i))) for i in range(n)])
    with make(nx, ny, None, obst) as one:                 # one process restores all rows
        one.load_rows(0, rec)
        one.run(b)
        assert np.array_equal(bits(one.save_rows()), bits(rec_ref)) and one.digest() == dig_ref
    if n >= 3:
        m = n - 1
        r = _launch(tmp_path, m, "load", nx, ny, a, b)
        assert r.returncode == 0, r.stdout[-4000:]
        got = np.concatenate([np.load(str(tmp_path / ("final_%d.npy" % i))) for i in range(m)])
        assert np.array_equal(bits(got), bits(rec_ref))
        for i in range(m):
            msg = (tmp_path / ("refused_%d.txt" % i)).read_text()
            assert "loaded into this slab handle with lbm_gpu_load_rows" in msg and "lbm_gpu_ipc_prepare" in msg, msg
    else:
        r = _launch(tmp_path, n, "load", nx, ny, a, b)      # same rank count, new processes
        assert r.returncode == 0, r.stdout[-4000:]
        got = np.concatenate([np.load(str(tmp_path / ("final_%d.npy" % i))) for i in range(n)])
        assert np.array_equal(bits(got), bits(rec_ref))
        for i in range(n):
            msg = (tmp_path / ("refused_%d.txt" % i)).read_text()
            assert "loaded into this slab handle with lbm_gpu_load_rows" in msg and "lbm_gpu_ipc_prepare" in msg, msg


# ------------------------------------------------------------------------------------------- CLI
def cli(cwd, params, env_extra):
    env = dict(os.environ)
    for k in ("LBM_CHECKPOINT", "LBM_CHECKPOINT_EVERY", "LBM_RESTART"):
        env.pop(k, None)
    env.update(env_extra)
    r = subprocess.run([EXE, params, os.path.join(ROOT, "inputs", "obstacles_128x128.dat")], cwd=str(cwd), env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    return r


def outputs(d):
    return [(d / n).read_bytes() for n in ("av_vels.dat", "final_state.dat")]


@pytest.mark.parametrize("knobs", [{}, {"LBM_PRECISION": "f64"}, {"LBM_PRECISION": "f16"}, {"LBM_STRICT": "1"}],
                         ids=["f32", "f64", "f16", "strict"])
def test_cli_restart_gives_the_uninterrupted_files(tmp_path, knobs):
    full_params = os.path.join(ROOT, "inputs", "input_128x128.params")
    lines = open(full_params).read().split("\n")
    assert lines[2] == "40000"
    lines[2] = "15000"
    short_params = tmp_path / "short.params"
    short_params.write_text("\n".join(lines))
    ref, part, every = tmp_path / "ref", tmp_path / "part", tmp_path / "every"
    for d in (ref, part, every):
        d.mkdir()
    r = cli(ref, full_params, knobs)
    assert r.returncode == 0, r.stderr
    ckpt = tmp_path / "run.ckpt"
    r = cli(part, str(short_params), dict(knobs, LBM_CHECKPOINT=str(ckpt)))
    assert r.returncode == 0, r.stderr
    assert "Elapsed Checkpoint time:" in r.stdout
    r = cli(part, full_params, dict(knobs, LBM_RESTART=str(ckpt)))
    assert r.returncode == 0, r.stderr
    assert outputs(part) == outputs(ref)
    # periodic checkpoints cut the run into lbm_gpu_run calls: no output bit changes, no .tmp is left
    ck2 = every / "every.ckpt"
    r = cli(every, str(short_params), dict(knobs, LBM_CHECKPOINT=str(ck2), LBM_CHECKPOINT_EVERY="4000"))
    assert r.returncode == 0, r.stderr
    assert ck2.read_bytes() == ckpt.read_bytes()
    # the restart may split the rows over another number of GPUs (binary16 lattices are single-GPU)
    gpus = 1 if knobs.get("LBM_PRECISION") == "f16" else min(2, L.load_library().lbm_gpu_device_count())
    r = cli(every, full_params, dict(knobs, LBM_RESTART=str(ck2), LBM_CHECKPOINT=str(ck2), LBM_CHECKPOINT_EVERY="7001",
                                     LBM_GPUS=str(gpus)))
    assert r.returncode == 0, r.stderr
    assert outputs(every) == outputs(ref)
    assert sorted(os.listdir(str(every))) == ["av_vels.dat", "every.ckpt", "final_state.dat"]


def test_cli_restart_catches_a_flipped_lattice_byte(tmp_path):
    short = tmp_path / "short.params"
    lines = open(os.path.join(ROOT, "inputs", "input_128x128.params")).read().split("\n")
    lines[2] = "300"
    short.write_text("\n".join(lines))
    ckpt = tmp_path / "run.ckpt"
    r = cli(tmp_path, str(short), {"LBM_CHECKPOINT": str(ckpt)})
    assert r.returncode == 0, r.stderr
    data = bytearray(ckpt.read_bytes())
    data[96 + 300 * 4 + 1234 * 36 + 5] ^= 0x10        # one byte of cell 1234's speed 1
    bad = tmp_path / "bad.ckpt"
    bad.write_bytes(bytes(data))
    out = tmp_path / "out"
    out.mkdir()
    r = cli(out, os.path.join(ROOT, "inputs", "input_128x128.params"), {"LBM_RESTART": str(bad)})
    assert r.returncode == 1 and "checksum differs from the one in its header: the file is corrupt" in r.stderr
    assert os.listdir(str(out)) == []
