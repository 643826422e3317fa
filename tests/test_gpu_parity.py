"""GPU parity tests: the CUDA path, called through the C-ABI (include/lbm_gpu.h), against
the CPU oracle on the same seeded inputs.

Bar (tier rules + BASELINE.json north_star):
  * LBM_GPU_STRICT build of the kernel (source operation order, no FMA): BIT-EXACT
    lattice after k steps against the oracle (which itself is bit-exact against the
    reference compiled with -O2 -ffp-contract=off, tests/test_oracle_vs_reference.py);
  * default (FMA-contracted) kernel: relative difference per speed <= 2e-5 after 50
    steps -- float arithmetic, so not bit-exact; the reference's own -Ofast build
    differs from its -O2 build by the same order (SURVEY.md section 7, "fp32 chaos");
  * av_vels: |gpu - oracle(double accumulation)| <= 1e-6 relative (strict: 1e-7).
"""
import numpy as np
import pytest

import lbm_b200 as L
import oracle_lib as O
import readout_ref as R

pytestmark = pytest.mark.gpu

DENSITY, ACCEL, OMEGA = 0.1, 0.005, 1.85

SHAPES = [
    (128, 128), (128, 256), (256, 64), (64, 7), (4, 2), (8, 3), (36, 5), (132, 9),
    (1024, 17), (2048, 6), (1540, 12),
]
ODD_SHAPES = [(1, 2), (2, 3), (3, 5), (5, 4), (37, 11), (129, 4), (250, 9), (33, 2), (127, 3), (130, 5), (515, 4)]


def cluster_fits(nx, ny):
    """K6 keeps the double-buffered lattice in the shared memory of one 16-CTA cluster."""
    return 2 * 9 * ((ny + 15) // 16) * nx * 4 <= 227 * 1024


def _kernels_for(nx, ny=None, f64=False):
    ks = [L.KERNEL_SCALAR, L.KERNEL_PERSISTENT, L.KERNEL_VEC4]
    if not f64:
        ks.append(L.KERNEL_TMA)
        if ny is not None and cluster_fits(nx, ny):
            ks.append(L.KERNEL_CLUSTER)
    return ks


@pytest.mark.parametrize("nx,ny", SHAPES + ODD_SHAPES)
@pytest.mark.parametrize("steps", [1, 2, 10])
def test_strict_bit_exact(nx, ny, steps):
    cells, obst = O.random_lattice(nx, ny, seed=nx * 1000 + ny)
    ref, av_ref, av_ref_d = O.run(cells, obst, steps, DENSITY, ACCEL, OMEGA)
    for k in _kernels_for(nx, ny):
        with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=L.STRICT | k) as lat:
            av = lat.run(steps)
            got = lat.download()
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), \
            "kernel %d %dx%d: %d cells differ" % (k, nx, ny, np.count_nonzero((got != ref).any(axis=2)))
        np.testing.assert_allclose(av.astype(np.float64), av_ref_d, rtol=1e-7, atol=0)


@pytest.mark.parametrize("nx,ny", [(128, 128), (256, 64), (132, 9), (37, 11)])
def test_fast_kernel_tolerance(nx, ny):
    steps = 50
    cells, obst = O.random_lattice(nx, ny, seed=7)
    ref, _, av_ref_d = O.run(cells, obst, steps, DENSITY, ACCEL, OMEGA)
    for k in _kernels_for(nx, ny):
        with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=k) as lat:
            av = lat.run(steps)
            got = lat.download()
        rel = np.abs(got.astype(np.float64) - ref) / np.abs(ref)
        assert rel.max() <= 2e-5, "kernel %d: max rel %.3g" % (k, rel.max())
        np.testing.assert_allclose(av.astype(np.float64), av_ref_d, rtol=1e-5, atol=0)


def test_rest_state_and_obstacle_bits():
    """cells=NULL generates the reference's rest state on the device (d2q9-bgk.c:2802-2823);
    the packed-bit obstacle format gives the same lattice as the int array."""
    nx, ny = 256, 32
    _, obst = O.random_lattice(nx, ny, seed=3)
    cells = O.rest_cells(nx, ny, DENSITY)
    ref, _, _ = O.run(cells, obst, 5, DENSITY, ACCEL, OMEGA)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, obstacles=obst, flags=L.STRICT) as lat:
        assert np.array_equal(lat.download(), cells)
        lat.run(5)
        a = lat.download()
        assert lat.info().free_cells == int((obst == 0).sum())
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, obstacles=L.pack_obstacle_bits(obst), bits=True,
                   flags=L.STRICT) as lat:
        lat.run(5)
        b = lat.download()
    assert np.array_equal(a, ref)
    assert np.array_equal(b, ref)


@pytest.mark.parametrize("kernel", ["vec4", "persistent", "scalar", "tma", "cluster"])
def test_chunked_runs_equal_one_run(kernel):
    """run(a); run(b) == run(a+b): no state is lost between calls (odd and even splits)."""
    k = {"vec4": L.KERNEL_VEC4, "persistent": L.KERNEL_PERSISTENT, "scalar": L.KERNEL_SCALAR, "tma": L.KERNEL_TMA,
         "cluster": L.KERNEL_CLUSTER}[kernel]
    nx, ny = 128, 24
    cells, obst = O.random_lattice(nx, ny, seed=11)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=k) as lat:
        av_all = lat.run(9)
        one = lat.download()
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=k) as lat:
        av_parts = np.concatenate([lat.run(1), lat.run(3), lat.run(0), lat.run(5)])
        parts = lat.download()
    assert np.array_equal(one, parts)
    assert np.array_equal(av_all, av_parts)


def test_long_runs_are_segmented_transparently():
    """More steps than one run segment (65536): same av_vels and lattice as several calls."""
    nx, ny, steps = 32, 8, 70000
    cells, obst = O.random_lattice(nx, ny, seed=19, p_obst=0.05)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst) as lat:
        av = lat.run(steps)
        one = lat.download()
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst) as lat:
        parts = np.concatenate([lat.run(30000), lat.run(40000)])
        two = lat.download()
    assert av.shape == (steps,) and np.array_equal(av, parts) and np.array_equal(one, two)
    assert np.all(np.isfinite(av))


def test_kernel_selection():
    """Small single-GPU grids take the persistent kernel, big ones one launch per step,
    widths that are not a multiple of 4 the scalar kernel; all give the same bits."""
    with L.Lattice(128, 128, DENSITY, ACCEL, OMEGA) as lat:
        assert lat.info().kernel == L.KERNEL_PAIRS               # lives in L2, two timesteps per barrier (test_gpu_pairs.py)
    with L.Lattice(640, 512, DENSITY, ACCEL, OMEGA) as lat:
        assert lat.info().kernel == L.KERNEL_PERSISTENT          # lives in L2
    with L.Lattice(128, 128, DENSITY, ACCEL, OMEGA, flags=L.KERNEL_CLUSTER) as lat:
        assert lat.info().kernel == L.KERNEL_CLUSTER             # opt-in: lives in one cluster's DSMEM
    with L.Lattice(130, 16, DENSITY, ACCEL, OMEGA) as lat:
        assert lat.info().kernel == L.KERNEL_PERSISTENT          # one cell per thread
    with L.Lattice(4098, 4096, DENSITY, ACCEL, OMEGA) as lat:
        assert lat.info().kernel == L.KERNEL_VEC4                # any width
    with L.Lattice(4096, 4096, DENSITY, ACCEL, OMEGA) as lat:
        assert lat.info().kernel == L.KERNEL_TB2                 # two timesteps per pass (tests/test_gpu_tb2.py)
    nx, ny = 1024, 600          # more tiles than resident blocks: every block loops
    cells, obst = O.random_lattice(nx, ny, seed=13, p_obst=0.01)
    res = []
    for k in (L.KERNEL_VEC4, L.KERNEL_PERSISTENT):
        with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=k) as lat:
            av = lat.run(7)
            res.append((lat.download(), av))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])


def test_final_fields_and_av_velocity():
    nx, ny = 128, 20
    cells, obst = O.random_lattice(nx, ny, seed=5)
    ref, _, _ = O.run(cells, obst, 3, DENSITY, ACCEL, OMEGA)
    ux, uy, u, pr = O.final_state(ref, obst, DENSITY)
    _, tot, n = O.av_velocity(ref, obst)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=L.STRICT) as lat:
        lat.run(3)
        gux, guy, gu, gpr = lat.final_fields()
        assert np.array_equal(gux, ux) and np.array_equal(guy, uy)
        assert np.array_equal(gu, u) and np.array_equal(gpr, pr)
        # a row range
        sub = lat.final_fields(row0=5, nrows=7)
        assert np.array_equal(sub[3], pr[5:12])
        assert abs(lat.av_velocity() - tot / n) <= 1e-7 * (tot / n)
        assert lat.av_velocity() == R.host_average(R.fixed_u_sum(u, obst), n, np.float32)   # exact sum
        rows = lat.download_rows(4, 3)
        assert np.array_equal(rows, ref[4:7])


def test_upload_round_trip():
    nx, ny = 64, 8
    cells, obst = O.random_lattice(nx, ny, seed=2)
    other, _ = O.random_lattice(nx, ny, seed=99)
    ref, _, _ = O.run(other, obst, 3, DENSITY, ACCEL, OMEGA)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=L.STRICT) as lat:
        lat.run(1)                       # odd parity, then replace the lattice
        lat.upload(other)
        assert np.array_equal(lat.download(), other)
        lat.run(3)
        assert np.array_equal(lat.download(), ref)


def test_f64_kernel_matches_f64_oracle():
    nx, ny = 128, 16
    cells, obst = O.random_lattice(nx, ny, seed=4, dtype=np.float64)
    ref, av_ref, _ = O.run(cells, obst, 10, DENSITY, ACCEL, OMEGA)
    for k in (L.KERNEL_SCALAR, L.KERNEL_VEC4, L.KERNEL_PERSISTENT):
        with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, f64=True,
                       flags=L.STRICT | k) as lat:
            av = lat.run(10)
            got = lat.download()
        assert np.array_equal(got, ref)
        np.testing.assert_allclose(av, av_ref, rtol=1e-12)


def test_mass_is_conserved_over_many_steps():
    """total_density (d2q9-bgk.c:2900-2916) stays constant: propagate moves, rebound swaps,
    BGK conserves mass, accelerate_flow adds what it removes."""
    nx, ny = 256, 128
    _, obst = O.random_lattice(nx, ny, seed=8, p_obst=0.02)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, obstacles=obst) as lat:
        m0 = lat.download().astype(np.float64).sum()
        av = lat.run(2000)
        m1 = lat.download().astype(np.float64).sum()
    assert abs(m1 - m0) / m0 < 2e-5
    assert np.all(np.isfinite(av)) and np.all(av > 0)


def test_blown_up_lattice_reports_nan_like_the_reference():
    """A lattice with a zero-density cell makes the reference's float sum NaN from that step
    on (0/0 in the velocity); the exact integer sum cannot hold NaN, so the kernel marks
    the step instead and the host reports NaN -- check.py then fails the run as it would
    fail the reference's."""
    nx, ny = 64, 8
    cells, obst = O.random_lattice(nx, ny, seed=6, p_obst=0.0, walls=False)
    obst[:] = 0
    cells[3, 10, :] = 0.0
    cells[2:5, 9:12, :] = 0.0            # a hole of zero density: pulled values are all zero
    for k in (L.KERNEL_VEC4, L.KERNEL_SCALAR, L.KERNEL_PERSISTENT, L.KERNEL_TMA, L.KERNEL_CLUSTER):
        with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=obst, flags=k) as lat:
            av = lat.run(3)
        assert np.isnan(av[0]), (k, av)
    _, av_ref, _ = O.run(cells, obst, 1, DENSITY, ACCEL, OMEGA)
    assert np.isnan(av_ref[0])


@pytest.mark.parametrize("density,accel,omega", [(0.1, 1.2, 1.85), (0.3, 0.9, 1.0), (0.05, 2.5, 0.6), (1.0, 0.001, 1.99)])
def test_other_parameters_and_the_accelerate_guard(density, accel, omega):
    """Parameters far from the shipped ones; with a large accel the guard of accelerate_flow
    (d2q9-bgk.c:247-249) is false for part of row ny-2.  Every kernel, one slab and three."""
    nx, ny, steps = 132, 9, 4
    cells, obst = O.random_lattice(nx, ny, seed=31, density=density)
    ref, _, av_ref = O.run(cells, obst, steps, density, accel, omega)
    for k in _kernels_for(nx, ny):
        for n in ((1, 3) if k not in (L.KERNEL_PERSISTENT, L.KERNEL_CLUSTER) else (1,)):
            with L.Lattice(nx, ny, density, accel, omega, cells=cells, obstacles=obst, flags=L.STRICT | k,
                           n_gpus=n, device_ids=[0] * n) as lat:
                av = lat.run(steps)
                assert np.array_equal(lat.download().view(np.uint32), ref.view(np.uint32)), (k, n)
            ok = np.isfinite(av_ref)
            np.testing.assert_allclose(av[ok].astype(np.float64), av_ref[ok], rtol=1e-6)


def test_degenerate_masks():
    """No obstacle file at all (obstacles=NULL), and a grid that is all obstacles: the
    reference divides by tot_cells = 0 there (d2q9-bgk.c:1811) and gets NaN; so do we."""
    nx, ny = 64, 6
    cells, _ = O.random_lattice(nx, ny, seed=12)
    none = np.zeros((ny, nx), dtype=np.int32)
    ref, _, av_ref = O.run(cells, none, 4, DENSITY, ACCEL, OMEGA)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=None, flags=L.STRICT) as lat:
        av = lat.run(4)
        assert np.array_equal(lat.download(), ref)
        assert lat.info().free_cells == nx * ny
    np.testing.assert_allclose(av, av_ref, rtol=1e-6)
    full = np.ones((ny, nx), dtype=np.int32)
    ref, _, _ = O.run(cells, full, 3, DENSITY, ACCEL, OMEGA)
    with L.Lattice(nx, ny, DENSITY, ACCEL, OMEGA, cells=cells, obstacles=full, flags=L.STRICT) as lat:
        av = lat.run(3)
        assert np.array_equal(lat.download(), ref)          # pure bounce-back everywhere
        assert lat.info().free_cells == 0
    assert np.all(np.isnan(av))


def test_errors_are_reported_not_fatal():
    with pytest.raises(L.LbmError, match="ny >= 2"):
        L.Lattice(8, 1, DENSITY, ACCEL, OMEGA)
    with pytest.raises(L.LbmError, match="single precision only"):
        L.Lattice(16, 4, DENSITY, ACCEL, OMEGA, flags=L.KERNEL_TMA, f64=True)
    with pytest.raises(L.LbmError, match="fits in one cluster"):
        L.Lattice(2048, 2048, DENSITY, ACCEL, OMEGA, flags=L.KERNEL_CLUSTER)
    with L.Lattice(8, 4, DENSITY, ACCEL, OMEGA) as lat:
        with pytest.raises(L.LbmError, match="double precision|single precision"):
            L.load_library().lbm_gpu_run_f64(lat.h, 1, None) and L.binding._check(1)
        with pytest.raises(L.LbmError, match="not held"):
            lat.download_rows(3, 5)
