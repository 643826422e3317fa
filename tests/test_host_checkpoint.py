"""LBM_RESTART checks a checkpoint against the run's inputs before the GPU is touched: each
mismatch ends in die() with a message that names it, and no output file is written.  These
paths end before lbm_gpu_create, so they run on CPU.  The file layout is the one documented in
advanced-hpc-lbm_b200/host/lbm_io.h."""
import os
import struct
import subprocess

import numpy as np
import pytest

import lbm_b200 as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "d2q9-bgk")
PARAMS = os.path.join(ROOT, "inputs", "input_128x128.params")
OBST = os.path.join(ROOT, "inputs", "obstacles_128x128.dat")

pytestmark = pytest.mark.skipif(not os.path.exists(EXE) or not os.path.exists(PARAMS),
                                reason="host binary or shipped inputs not built (make)")

KIND = {"f32": 0, "f64": 1, "f16": 2}
RECORD = {"f32": 36, "f64": 72, "f16": 18}
AV = {"f32": 4, "f64": 8, "f16": 4}


def read_obstacles(path, nx, ny):
    obst = np.zeros((ny, nx), dtype=np.int32)
    for line in open(path):
        if line.strip():
            x, y, _ = map(int, line.split())
            obst[y, x] = 1
    return obst


def obstacle_hash(obst):
    """lbm_obstacle_hash: FNV-1a over the 32-bit words of the packed mask."""
    h = 0xcbf29ce484222325
    for w in L.pack_obstacle_bits(obst).ravel():
        h = ((h ^ int(w)) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


def header(nx=128, ny=128, reynolds_dim=10, density="0.1", accel="0.005", omega="1.85", kind="f32", strict=0,
           t=100, ohash=None, magic=b"LBMCKPT\0", version=1, checksum=0):
    f32 = [struct.unpack("<I", struct.pack("<f", float(v)))[0] for v in (density, accel, omega)]
    f64 = [struct.unpack("<Q", struct.pack("<d", float(v)))[0] for v in (density, accel, omega)]
    if ohash is None:
        ohash = obstacle_hash(read_obstacles(OBST, 128, 128))
    return (magic + struct.pack("<IIIiii", version, KIND[kind], strict, nx, ny, reynolds_dim)
            + struct.pack("<IIII", *f32, 0) + struct.pack("<QQQ", *f64) + struct.pack("<qQQ", t, ohash, checksum))


def write_checkpoint(path, hdr_kw=None, kind="f32", t=100, trim=0, nx=128, ny=128):
    kw = dict(kind=kind, t=t, nx=nx, ny=ny)
    kw.update(hdr_kw or {})
    body = header(**kw)
    assert len(body) == 96
    size = 96 + t * AV[kind] + ny * nx * RECORD[kind] - trim
    with open(path, "wb") as f:
        f.write(body)
        f.write(b"\0" * (size - 96))


def restart(tmp_path, ckpt, env=None, params=PARAMS, obst=OBST):
    e = dict(os.environ, LBM_RESTART=str(ckpt))
    e.update(env or {})
    r = subprocess.run([EXE, params, obst], cwd=str(tmp_path), env=e, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    outputs = [n for n in ("av_vels.dat", "final_state.dat") if (tmp_path / n).exists()]
    return r.returncode, r.stderr, outputs


CASES = [
    ("magic", dict(magic=b"NOTACKPT"), {}, "not a checkpoint of this program (wrong magic)"),
    ("version", dict(version=2), {}, "format version 2, this program reads version 1"),
    ("nx", dict(nx=64), {}, "nx is 64, the parameter file's is 128"),
    ("ny", dict(ny=256), {}, "ny is 256, the parameter file's is 128"),
    ("reynolds_dim", dict(reynolds_dim=11), {}, "reynolds_dim is 11, the parameter file's is 10"),
    ("density", dict(density="0.1000001"), {}, "density differs from the parameter file's"),
    ("accel", dict(accel="0.006"), {}, "accel differs from the parameter file's"),
    ("omega", dict(omega="1.7"), {}, "omega differs from the parameter file's"),
    ("obstacles", dict(ohash=12345), {}, "written with another obstacle file"),
    ("precision-f64", dict(kind="f64"), {}, "holds a fp64 (LBM_PRECISION=f64) lattice, this run asks for fp32"),
    ("precision-f16", dict(), {"LBM_PRECISION": "f16"}, "holds a fp32 lattice, this run asks for binary16"),
    ("strict", dict(strict=1), {}, "written with LBM_STRICT=1, this run has LBM_STRICT=0"),
    ("not-strict", dict(), {"LBM_STRICT": "1"}, "written with LBM_STRICT=0, this run has LBM_STRICT=1"),
    ("beyond-maxIters", dict(t=40001), {}, "is at step 40001, beyond maxIters = 40000"),
]


@pytest.mark.parametrize("name,hdr,env,msg", CASES, ids=[c[0] for c in CASES])
def test_restart_refuses_a_mismatched_header(tmp_path, name, hdr, env, msg):
    ckpt = tmp_path / "run.ckpt"
    kind = hdr.get("kind", "f32")
    t = hdr.get("t", 100)
    write_checkpoint(ckpt, {k: v for k, v in hdr.items() if k not in ("kind", "t")}, kind=kind,
                     t=t if t <= 40000 else 100, nx=hdr.get("nx", 128), ny=hdr.get("ny", 128))
    if t > 40000:          # the header's t alone: the step check comes before the size check
        data = bytearray(ckpt.read_bytes())
        data[72:80] = struct.pack("<q", t)
        ckpt.write_bytes(bytes(data))
    rc, err, outputs = restart(tmp_path, ckpt, env)
    assert rc == 1 and err.startswith("Error at line "), err
    assert msg in err, err
    assert outputs == []


def test_restart_refuses_another_obstacle_file(tmp_path):
    """The header carries the hash of the obstacle mask the checkpoint was written with."""
    ckpt = tmp_path / "run.ckpt"
    write_checkpoint(ckpt)
    other = tmp_path / "obstacles.dat"
    other.write_text(open(OBST).read() + "5 5 1\n")
    rc, err, outputs = restart(tmp_path, ckpt, obst=str(other))
    assert rc == 1 and "written with another obstacle file" in err, err
    assert outputs == []


@pytest.mark.parametrize("trim", [1, 18 * 128, -4])
def test_restart_refuses_a_file_of_the_wrong_size(tmp_path, trim):
    ckpt = tmp_path / "run.ckpt"
    write_checkpoint(ckpt, trim=trim)
    rc, err, outputs = restart(tmp_path, ckpt)
    expect = 96 + 100 * 4 + 128 * 128 * 36
    assert rc == 1 and "file has %d bytes, its header implies %d" % (expect - trim, expect) in err, err
    assert outputs == []


def test_restart_refuses_a_truncated_header(tmp_path):
    ckpt = tmp_path / "run.ckpt"
    ckpt.write_bytes(header()[:40])
    rc, err, outputs = restart(tmp_path, ckpt)
    assert rc == 1 and "truncated header (40 of 96 bytes)" in err, err
    assert outputs == []


def test_restart_refuses_a_missing_file(tmp_path):
    rc, err, outputs = restart(tmp_path, tmp_path / "none.ckpt")
    assert rc == 1 and "could not open checkpoint file" in err, err
    assert outputs == []


def test_a_matching_header_passes_the_checks(tmp_path):
    """A header that matches gets past every check: what stops it is the device (none here) or,
    with a GPU, the lattice checksum of the zero-filled records."""
    ckpt = tmp_path / "run.ckpt"
    write_checkpoint(ckpt, dict(checksum=1))
    rc, err, outputs = restart(tmp_path, ckpt)
    assert rc == 1
    assert "no CUDA device available" in err or "checksum differs from the one in its header" in err, err
    assert outputs == []


@pytest.mark.parametrize("value", ["0", "-3", "x"])
def test_checkpoint_every_needs_a_positive_count(tmp_path, value):
    e = dict(os.environ, LBM_CHECKPOINT=str(tmp_path / "c"), LBM_CHECKPOINT_EVERY=value)
    r = subprocess.run([EXE, PARAMS, OBST], cwd=str(tmp_path), env=e, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1 and "LBM_CHECKPOINT_EVERY must be a positive number of steps" in r.stderr


def test_checkpoint_every_needs_a_path(tmp_path):
    e = dict(os.environ, LBM_CHECKPOINT_EVERY="10")
    e.pop("LBM_CHECKPOINT", None)
    r = subprocess.run([EXE, PARAMS, OBST], cwd=str(tmp_path), env=e, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1 and "LBM_CHECKPOINT_EVERY needs LBM_CHECKPOINT" in r.stderr
