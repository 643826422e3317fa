"""lbm_gpu_coarse_fields (Lattice.coarse_fields): block means of the fields computed on the GPU,
checked bit for bit against the CPU restatement in tests/coarse_ref.py, which starts from
final_fields (held exact by test_gpu_readout.py):

  * factors 1, 2, 3, 4, 7, 8, 16 and 256, fp32 and binary16 outputs, ragged shapes, fp32 and
    STORE_F16 lattices after steps with obstacles, a grid that takes several staging chunks;
  * three slabs on one device and two GPUs give the bits of one slab, also for coarse rows cut
    by a slab boundary; slab handles serve the coarse rows they hold and refuse the others;
  * a NaN or out-of-range cell makes only its own block's affected fields NaN;
  * every refusal writes nothing, and a call changes neither the lattice nor the run.
"""
import numpy as np
import pytest

import coarse_ref as CR
import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85
FACTORS = [1, 2, 3, 4, 7, 8, 16, 256]


def same(a, b):
    """Equal bit for bit, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    u = {2: np.uint16, 4: np.uint32}[a.dtype.itemsize]
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(u), b[~nb].view(u))


def check_all(lat, factors=FACTORS):
    fields = lat.final_fields()
    for factor in factors:
        for f16 in (False, True):
            got = lat.coarse_fields(factor, f16=f16)
            want = CR.coarse_fields(fields, factor, D, f16=f16)
            for k in range(4):
                assert same(got[k], want[k]), (factor, f16, k)


def make(nx, ny, seed, f16_store=False, slabs=1, p_obst=0.1, device_ids=None):
    cells, obst = O.random_lattice(nx, ny, seed=seed, p_obst=p_obst)
    return L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, n_gpus=slabs,
                     device_ids=device_ids or [0] * slabs, flags=L.STORE_F16 if f16_store else 0)


SHAPES = [(300, 70), (1, 50), (5, 3), (257, 259), (64, 64), (1000, 9)]


@pytest.mark.parametrize("store", ["f32", "f16"])
@pytest.mark.parametrize("nx,ny", SHAPES)
def test_exact_against_the_restatement(nx, ny, store):
    with make(nx, ny, seed=nx + ny, f16_store=(store == "f16")) as lat:
        lat.run(5)
        check_all(lat)


def test_several_staging_chunks():
    """8190 x 2600: factor 1 / F16 takes 6 chunks of 512 rows, factor 2 / F32 three of 512
    coarse rows, factor 3 / F32 two of 768; one slab and three."""
    nx, ny = 8190, 2600
    for slabs in (1, 3):
        with make(nx, ny, seed=7, slabs=slabs) as lat:
            lat.run(2)
            check_all(lat, factors=[1, 2, 3, 8])


def test_factor_one():
    with make(300, 70, seed=1) as lat:
        lat.run(3)
        fields = lat.final_fields()
        for a, b in zip(lat.coarse_fields(1), fields):
            assert same(a, b)
        h = lat.coarse_fields(1, f16=True)
        for k in range(3):
            assert same(h[k], fields[k].astype(np.float16))
        assert same(h[3], (fields[3] - CR.p0(D)).astype(np.float16))
        # decoded, the pressure is within binary16's 11 bits of its distance from p0 (and within
        # half of binary16's smallest spacing, 2^-24, plus the fp32 add, close to p0)
        err = np.abs(CR.decode_pressure(h[3], D) - fields[3])
        assert np.all(err <= np.abs(fields[3] - CR.p0(D)) * 2.0 ** -11 + 2.0 ** -24)


# ---------------------------------------------------------------------------- slabs
def test_three_slabs_on_one_device_give_the_bits_of_one():
    nx, ny = 97, 100                                   # slabs of 34, 33, 33 rows: boundaries 34 and 67
    cells, obst = O.random_lattice(nx, ny, seed=5, p_obst=0.1)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst) as one, \
            L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, n_gpus=3, device_ids=[0, 0, 0]) as three:
        assert three.info().n_gpus == 3
        one.run(4)
        three.run(4)
        assert one.digest() == three.digest()
        for factor in FACTORS + [5, 33, 34, 67]:
            for f16 in (False, True):
                a, b = one.coarse_fields(factor, f16=f16), three.coarse_fields(factor, f16=f16)
                for k in range(4):
                    assert same(a[k], b[k]), (factor, f16, k)
                ncy = a[0].shape[0]
                for crow0, n in ((0, 1), (ncy // 3, 2), (ncy - 1, 1)):
                    if crow0 + n <= ncy:
                        part = three.coarse_fields(factor, f16=f16, crow0=crow0, ncrows=n)
                        for k in range(4):
                            assert same(part[k], a[k][crow0:crow0 + n]), (factor, crow0, n)
        check_all(three)


def test_two_gpus_give_the_bits_of_one():
    if L.load_library().lbm_gpu_device_count() < 2:
        pytest.skip("needs two GPUs")
    nx, ny = 256, 101
    cells, obst = O.random_lattice(nx, ny, seed=9, p_obst=0.1)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst) as one, \
            L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, n_gpus=2, device_ids=[0, 1]) as two:
        one.run(6)
        two.run(6)
        for factor in (1, 2, 3, 8, 16, 256):
            for f16 in (False, True):
                a, b = one.coarse_fields(factor, f16=f16), two.coarse_fields(factor, f16=f16)
                for k in range(4):
                    assert same(a[k], b[k]), (factor, f16, k)


def test_slab_handles_serve_the_rows_they_hold():
    nx, ny = 120, 50
    cells, obst = O.random_lattice(nx, ny, seed=11, p_obst=0.1)
    sentinel = 7.0
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst) as whole:
        for r0, k in ((0, 24), (24, 26), (10, 30)):
            with L.Lattice(nx, ny, D, A, W, cells=cells[r0:r0 + k], obstacles=obst[r0:r0 + k], slab=(r0, k),
                           device_ids=[0]) as s:
                for factor in (1, 2, 3, 4, 8, 16):
                    for f16 in (False, True):
                        crow0, n = s.coarse_rows(factor)
                        want = whole.coarse_fields(factor, f16=f16)
                        got = s.coarse_fields(factor, f16=f16)
                        assert got[0].shape[0] == n
                        for g, w in zip(got, want):
                            assert same(g, w[crow0:crow0 + n]), (r0, k, factor, f16)
                        # the coarse rows just outside what the slab holds entirely are refused
                        ncy = -(-ny // factor)
                        dt = np.float16 if f16 else np.float32
                        for bad in (crow0 - 1, crow0 + n):
                            if 0 <= bad < ncy:
                                out = [np.full((1, -(-nx // factor)), sentinel, dtype=dt) for _ in range(4)]
                                with pytest.raises(L.LbmError, match="coarse row %d " % bad):
                                    s.coarse_fields(factor, f16=f16, crow0=bad, ncrows=1, out=out)
                                assert all(np.all(o == dt(sentinel)) for o in out)


# ------------------------------------------------------------------------------ NaN
def test_nan_and_out_of_range_cells_mark_only_their_block():
    nx, ny, factor = 64, 40, 8
    cells, obst = O.random_lattice(nx, ny, seed=13, p_obst=0.0, walls=False)
    cells[3, 10, :] = np.nan                         # block (0, 1): every field NaN
    cells[20, 50, :] = 0.0                           # block (2, 6): |u_x| = 2 / 2^-15 = 2^16, rho finite
    cells[20, 50, 1], cells[20, 50, 3] = np.float32(1.0), np.float32(-1.0 + 2.0 ** -15)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst) as lat:
        fields = lat.final_fields()
        assert abs(fields[0][20, 50]) >= 2 ** 15 and np.isfinite(fields[0][20, 50])
        for f16 in (False, True):
            got = lat.coarse_fields(factor, f16=f16)
            want = CR.coarse_fields(fields, factor, D, f16=f16)
            nan = [np.isnan(g) for g in got]
            for k in range(4):
                assert same(got[k], want[k])
                assert nan[k][0, 1]
            assert nan[0][2, 6] and nan[2][2, 6] and not nan[1][2, 6] and not nan[3][2, 6]
            for k in range(4):
                nan[k][0, 1] = nan[k][2, 6] = False
                assert not nan[k].any()


# ------------------------------------------------------------------ refusals, effects
def test_refusals_write_nothing_and_change_nothing():
    nx, ny = 100, 30
    lib = L.load_library()
    with make(nx, ny, seed=17) as lat:
        lat.run(3)
        before = (lat.digest(), lat.info().steps_done, lat.info().kernel)
        for args, msg in (((0, 0), "factor"), ((257, 0), "factor"), ((2, 2), "format"),
                          ((2, 0, 0, -1), "negative"), ((2, 0, -1, 1), "coarse rows"),
                          ((2, 0, 14, 2), "coarse rows"), ((4, 1, 8, 1), "coarse rows")):
            factor, fmt = args[0], args[1]
            crow0, n = (args[2], args[3]) if len(args) > 2 else (0, 1)
            out = [np.full((2, nx), 7.0, dtype=np.float32) for _ in range(4)]
            rc = lib.lbm_gpu_coarse_fields(lat.h, factor, fmt, crow0, n, *[L.binding._ptr(o) for o in out])
            assert rc != 0, args
            assert msg in lib.lbm_gpu_last_error().decode(), (args, lib.lbm_gpu_last_error())
            assert all(np.all(o == 7.0) for o in out), args
        # ncrows = 0 succeeds and writes nothing
        for crow0 in (0, 7, 15, 99):
            out = [np.full((2, nx), 7.0, dtype=np.float32) for _ in range(4)]
            lat.coarse_fields(2, crow0=crow0, ncrows=0, out=out)
            assert all(np.all(o == 7.0) for o in out)
        assert (lat.digest(), lat.info().steps_done, lat.info().kernel) == before
    cells, obst = O.random_lattice(nx, ny, seed=17, dtype=np.float64)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, f64=True) as lat64:
        out = [np.full((2, nx), 7.0, dtype=np.float32) for _ in range(4)]
        with pytest.raises(L.LbmError, match="double-precision"):
            lat64.coarse_fields(2, out=out)
        assert all(np.all(o == 7.0) for o in out)


@pytest.mark.parametrize("store", ["f32", "f16"])
def test_a_call_between_runs_changes_nothing(store):
    nx, ny = 512, 300
    with make(nx, ny, seed=19, f16_store=(store == "f16")) as a, \
            make(nx, ny, seed=19, f16_store=(store == "f16")) as b:
        av_a = list(a.run(7))
        d0 = a.digest()
        for factor in (1, 4, 7):
            for f16 in (False, True):
                a.coarse_fields(factor, f16=f16)
        assert a.digest() == d0 and a.info().steps_done == 7
        av_a += list(a.run(8))
        av_b = b.run(15)
        assert same(np.array(av_a, dtype=np.float32), av_b)
        assert same(a.download(), b.download())
        assert a.info().kernel == b.info().kernel
