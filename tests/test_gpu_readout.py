"""The read-outs a user's results pass through -- final_fields (final_state.dat), av_velocity
(the Reynolds number), digest (LBM_DEBUG and the full-size comparisons), download,
download_rows, upload and the obstacle mask -- against exact CPU restatements
(tests/readout_ref.py) rather than tolerances:

  * on grids large enough that every one of them runs over several chunks of the 64 MiB
    staging buffer, with ragged last chunks, ranges that start inside a chunk and ranges across
    slab boundaries; fp32, fp64 and STORE_F16, one slab and three on one device;
  * av_vels of every strict kernel bit for bit, including K11 (run_batch) and both f16 kernels;
  * NaN, zero-density and blown-up cells: av_velocity and total_density report NaN;
  * row ranges at and beyond the edges of the grid.
"""
import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import lbm_b200 as L
import oracle_f16 as H
import oracle_lib as O
import readout_ref as R

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85


def same(a, b):
    """Equal bit for bit, except that any NaN equals any NaN (the device and the CPU make NaNs
    with different sign bits)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    u = np.uint64 if a.dtype == np.float64 else np.uint32
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(u), b[~nb].view(u))


def stored(cells, f16):
    """What the handle holds after create or upload with `cells`."""
    return H.f16_decode(H.f16_encode(cells, D), D) if f16 else cells


def make(cells, obst, kind, slabs, flags=0, bits=False):
    ny, nx, _ = cells.shape
    f = flags | (L.STORE_F16 if kind == "f16" else 0)
    mask = L.pack_obstacle_bits(obst) if bits else obst
    return L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=mask, f64=(kind == "f64"), flags=f, bits=bits,
                     n_gpus=slabs, device_ids=[0] * slabs)


def check_readouts(lat, want, obst, ranges):
    """Every read-out of the handle against the CPU restatement of the lattice `want`."""
    dtype = want.dtype.type
    ny = want.shape[0]
    held = lat.download()
    assert same(held, want)
    ref = O.final_state(want, obst, D)
    for field, r in zip(lat.final_fields(), ref):
        assert same(field, r)
    n = int((obst == 0).sum())
    assert lat.info().free_cells == n
    av = lat.av_velocity()
    assert same(dtype(av), R.host_average(R.fixed_u_sum(ref[2], obst), n, dtype)), av
    # the checksum of what the handle holds: that is `want` bit for bit, except that binary16
    # storage gives its NaNs the device's bit pattern
    d = lat.digest()
    want_d = (R.digest_mass(want), R.checksum(held))
    assert same(np.float64(d[0]), np.float64(want_d[0])) and d[1] == want_d[1], (d, want_d)
    for row0, nrows in ranges:
        assert 0 <= row0 and row0 + nrows <= ny
        for field, r in zip(lat.final_fields(row0, nrows), ref):
            assert same(field, r[row0:row0 + nrows]), (row0, nrows)
        if not lat.f64:
            assert same(lat.download_rows(row0, nrows), want[row0:row0 + nrows]), (row0, nrows)


def ragged_ranges(ny, chunk):
    """Row ranges that start inside a chunk, end inside one, cross one or more chunk boundaries,
    cross the boundaries of three slabs, or hold only the ragged last chunk."""
    third = ny // 3 + (1 if ny % 3 else 0)            # the first slab boundary of split_rows
    return [(0, 1), (1, chunk), (chunk - 3, 7), (chunk + 5, 2 * chunk + 11), (third - 9, 20),
            (third - chunk // 2, ny - third), (ny - ny % chunk - 1, ny % chunk + 1), (ny - 1, 1), (3, ny - 5)]


# (kind, nx, ny, slab counts, fields rows per chunk): 8190 x 2600 in fp32 is 11 field chunks
# of 256 rows with a ragged 40-row last one, 12 transfer chunks of 227 rows, and 3 int-mask
# chunks of 1024 rows whose last mask word per row is not full; fp64 halves the rows per chunk.
BIG = [("f32", 8190, 2600, 1, 256), ("f32", 8190, 2600, 3, 256), ("f16", 8190, 2600, 1, 256),
       ("f64", 8190, 1300, 1, 128), ("f64", 8190, 1300, 3, 128)]


@pytest.mark.parametrize("kind,nx,ny,slabs,chunk", BIG, ids=["%s-%dx%d-%dslab" % b[:4] for b in BIG])
def test_large_chunked_grids(kind, nx, ny, slabs, chunk):
    dtype = np.float64 if kind == "f64" else np.float32
    f16 = kind == "f16"
    cells, obst = O.random_lattice(nx, ny, seed=ny + slabs, dtype=dtype, p_obst=0.1)
    ranges = ragged_ranges(ny, chunk)
    with make(cells, obst, kind, slabs, flags=L.STRICT) as lat:
        assert lat.info().n_gpus == slabs
        check_readouts(lat, stored(cells, f16), obst, ranges)
        other, _ = O.random_lattice(nx, ny, seed=ny + slabs + 1, dtype=dtype)
        lat.upload(other)
        want = stored(other, f16)
        check_readouts(lat, want, obst, ranges[:3])
        del cells, other
        # one step and two: the lattice in either buffer
        for _ in range(2):
            av = lat.run(1)
            want, ref_av = R.strict_av_vels(want, obst, 1, D, A, W, f16=f16)
            assert lat.digest() == R.digest(want)
            assert same(av, ref_av)
        check_readouts(lat, want, obst, ranges[-2:])


def test_int_mask_and_bit_mask_read_out_the_same():
    """8192 x 2600: the int mask takes three staging chunks, the bit mask one."""
    nx, ny = 8192, 2600
    cells, obst = O.random_lattice(nx, ny, seed=41, p_obst=0.1)
    for slabs in (1, 3):
        for bits in (False, True):
            with make(cells, obst, "f32", slabs, flags=L.STRICT, bits=bits) as lat:
                check_readouts(lat, cells, obst, [(1023, 2), (2047, 553)])


# ------------------------------------------------------------------ av_vels bit for bit
SMALL = [(128, 128), (64, 24), (256, 37)]
STRICT_KERNELS = {"scalar": L.KERNEL_SCALAR, "vec4": L.KERNEL_VEC4, "tma": L.KERNEL_TMA,
                  "persistent": L.KERNEL_PERSISTENT, "cluster": L.KERNEL_CLUSTER, "pairs": L.KERNEL_PAIRS,
                  "tb2": L.KERNEL_TB2, "tb3": L.KERNEL_TB3}


@pytest.mark.parametrize("nx,ny", SMALL)
@pytest.mark.parametrize("steps", [1, 2, 5])
@pytest.mark.parametrize("kernel", list(STRICT_KERNELS))
def test_strict_av_vels_bit_for_bit(nx, ny, steps, kernel):
    cells, obst = O.random_lattice(nx, ny, seed=nx * 1000 + ny)
    ref, ref_av = R.strict_av_vels(cells, obst, steps, D, A, W)
    with make(cells, obst, "f32", 1, flags=L.STRICT | STRICT_KERNELS[kernel]) as lat:
        assert lat.info().kernel == STRICT_KERNELS[kernel]
        av = lat.run(steps)
        assert same(lat.download(), ref)
    assert same(av, ref_av), (av, ref_av)


@pytest.mark.parametrize("nx,ny", SMALL)
@pytest.mark.parametrize("kind,kernel", [("f32", L.KERNEL_VEC4), ("f32", L.KERNEL_SCALAR), ("f64", L.KERNEL_VEC4),
                                         ("f64", L.KERNEL_SCALAR), ("f16", L.KERNEL_VEC4), ("f16", L.KERNEL_TB2)])
def test_strict_av_vels_bit_for_bit_other_storage_and_slabs(nx, ny, kind, kernel):
    """fp64 and both f16 kernels (K1a-f16, K7-f16) on one slab; fp32 and fp64 on three."""
    steps = 5
    dtype = np.float64 if kind == "f64" else np.float32
    cells, obst = O.random_lattice(nx, ny, seed=nx + ny, dtype=dtype)
    ref, ref_av = R.strict_av_vels(cells, obst, steps, D, A, W, f16=(kind == "f16"))
    for slabs in ((1,) if kind == "f16" else (1, 3)):
        with make(cells, obst, kind, slabs, flags=L.STRICT | kernel) as lat:
            av = lat.run(steps)
            assert same(lat.download(), ref)
        assert same(av, ref_av), (slabs, av, ref_av)


@pytest.mark.parametrize("steps", [1, 2, 5])
def test_strict_av_vels_bit_for_bit_in_a_batch(steps):
    nx, ny = 128, 96
    lats, refs = [], []
    for i, (d, a, w) in enumerate([(0.1, 0.005, 1.85), (0.12, 0.004, 1.6), (0.09, 0.006, 1.0)]):
        cells, obst = O.random_lattice(nx, ny, seed=50 + i)
        refs.append(R.strict_av_vels(cells, obst, steps, d, a, w)[1])
        lats.append(L.Lattice(nx, ny, d, a, w, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_PAIRS))
    av = L.run_batch(lats, steps)
    for row, ref_av in zip(av, refs):
        assert same(row, ref_av), (row, ref_av)
    for lat in lats:
        lat.close()


@pytest.mark.parametrize("kind", ["f32", "f64", "f16"])
def test_default_build_read_outs_are_exact(kind):
    """The step kernels' default arithmetic is not the reference's, but final_fields and
    av_velocity read the lattice with the strict operation order in either build."""
    nx, ny = 256, 64
    dtype = np.float64 if kind == "f64" else np.float32
    cells, obst = O.random_lattice(nx, ny, seed=17, dtype=dtype)
    with make(cells, obst, kind, 1) as lat:
        lat.run(7)
        check_readouts(lat, lat.download(), obst, [(3, 40)])


@settings(max_examples=100, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large],
          derandomize=True)
@given(nx=st.integers(1, 300), ny=st.integers(2, 40), steps=st.integers(1, 7), seed=st.integers(0, 10 ** 6),
       p_obst=st.sampled_from([0.0, 0.02, 0.2, 0.6]),
       kernel=st.sampled_from([L.KERNEL_VEC4, L.KERNEL_SCALAR, L.KERNEL_PERSISTENT, L.KERNEL_TMA, L.KERNEL_CLUSTER]),
       slabs=st.integers(1, 4), density=st.sampled_from([0.1, 0.37]), accel=st.sampled_from([0.005, 0.05, 1.1]),
       omega=st.sampled_from([0.7, 1.0, 1.85]), walls=st.booleans())
def test_any_configuration_gives_the_exact_av_vels(nx, ny, steps, seed, p_obst, kernel, slabs, density, accel, omega,
                                                   walls):
    cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=p_obst, walls=walls)
    ref, ref_av = R.strict_av_vels(cells, obst, steps, density, accel, omega)
    n = 1 if kernel in (L.KERNEL_PERSISTENT, L.KERNEL_CLUSTER) else min(slabs, ny)
    with L.Lattice(nx, ny, density, accel, omega, cells=cells, obstacles=obst, flags=L.STRICT | kernel, n_gpus=n,
                   device_ids=[0] * n) as lat:
        av = lat.run(steps)
        got = lat.download()
        fields = lat.final_fields()
        av_now = lat.av_velocity()
    assert same(got, ref)
    assert same(av, ref_av), (av, ref_av)
    ref_fields = O.final_state(ref, obst, density)
    for a, b in zip(fields, ref_fields):
        assert same(a, b)
    assert same(np.float32(av_now), R.host_average(R.fixed_u_sum(ref_fields[2], obst), int((obst == 0).sum()),
                                                  np.float32))


# ---------------------------------------------------------------------------- NaN
def blown_up(kind, nx=300, ny=40):
    dtype = np.float64 if kind == "f64" else np.float32
    cells, obst = O.random_lattice(nx, ny, seed=6, dtype=dtype, p_obst=0.05)
    obst[2:6, 9:13] = 0
    cells[3, 10, :] = np.nan
    cells[2:5, 20:23, :] = 0.0                      # a hole of zero density: 0/0 in the velocity
    return cells, obst


@pytest.mark.parametrize("kind,slabs", [("f32", 1), ("f32", 3), ("f64", 1), ("f64", 3), ("f16", 1)])
def test_nan_and_zero_density_cells_read_out_nan(kind, slabs):
    cells, obst = blown_up(kind)
    want = stored(cells, kind == "f16")
    assert np.isnan(O.av_velocity(want, obst)[0])          # what the reference reports
    with make(cells, obst, kind, slabs) as lat:
        assert np.isnan(lat.av_velocity())
        mass, cs = lat.digest()
        assert np.isnan(mass)
        assert cs == R.checksum(want if kind != "f16" else lat.download())
        check_readouts(lat, want, obst, [(2, 5), (38, 2)])


@pytest.mark.parametrize("kind", ["f32", "f64", "f16"])
def test_a_cell_beyond_the_speed_limit_reads_out_nan(kind):
    """A finite cell with |u| >= LBM_SPEED_LIMIT: av_velocity is NaN, as run() reports such a
    step; the digest stays finite."""
    cells, obst = O.random_lattice(300, 40, seed=8, dtype=np.float64 if kind == "f64" else np.float32)
    obst[17, 30] = 0
    cells[17, 30, :] = 0.0
    cells[17, 30, 1], cells[17, 30, 3] = 0.5, -0.3          # rho 0.2, u_x 4
    want = stored(cells, kind == "f16")
    assert O.final_state(want, obst, D)[2][17, 30] >= R.SPEED_LIMIT
    with make(cells, obst, kind, 1) as lat:
        assert np.isnan(lat.av_velocity())
        assert np.isfinite(lat.digest()[0])
        check_readouts(lat, want, obst, [(17, 1)])
    obst[17, 30] = 1                                        # the same cell as an obstacle is not counted
    with make(cells, obst, kind, 1) as lat:
        assert np.isfinite(lat.av_velocity())
        check_readouts(lat, want, obst, [])


# -------------------------------------------------------------------------- edges
@pytest.mark.parametrize("kind,slabs", [("f32", 1), ("f32", 3), ("f64", 1)])
def test_row_range_edges(kind, slabs):
    nx, ny = 200, 30
    dtype = np.float64 if kind == "f64" else np.float32
    cells, obst = O.random_lattice(nx, ny, seed=3, dtype=dtype)
    lib = L.load_library()
    with make(cells, obst, kind, slabs) as lat:
        before = lat.digest()
        sentinel = [np.full((2, nx), 7.0, dtype=dtype) for _ in range(4)]
        # nrows = 0 succeeds and writes nothing, wherever it starts
        for row0 in (0, 5, ny):
            out = [s.copy() for s in sentinel]
            lat.final_fields(row0, 0, out=out)
            assert all(np.array_equal(o, s) for o, s in zip(out, sentinel))
            if kind != "f64":
                buf = np.full((2, nx, 9), 7.0, dtype=np.float32)
                L.binding._check(lib.lbm_gpu_download_rows(lat.h, row0, 0, L.binding._ptr(buf)))
                assert np.all(buf == 7.0)
        # a negative count, a negative start, a range past ny: refused, nothing written
        for row0, nrows in ((0, -1), (-1, 2), (ny - 1, 2), (ny, 1)):
            out = [s.copy() for s in sentinel]
            with pytest.raises(L.LbmError):
                lat.final_fields(row0, nrows, out=out)
            assert all(np.array_equal(o, s) for o, s in zip(out, sentinel)), (row0, nrows)
            if kind != "f64":
                buf = np.full((2, nx, 9), 7.0, dtype=np.float32)
                with pytest.raises(L.LbmError):
                    L.binding._check(lib.lbm_gpu_download_rows(lat.h, row0, nrows, L.binding._ptr(buf)))
                assert np.all(buf == 7.0), (row0, nrows)
            assert lat.digest() == before
        check_readouts(lat, cells, obst, [(ny - 2, 2), (0, ny)])
