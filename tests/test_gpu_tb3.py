"""K10, the three-timesteps-per-pass kernel (temporal blocking), through the C-ABI.

Three iterations of the reference's loop (d2q9-bgk.c:180-201) fused into one pass over HBM
must give what three separate iterations give:
  * strict build: the oracle's lattice bit for bit and its av_vels, for every remainder of
    the step count (a last pair of steps is done by K7, a last single step by K1a), any
    split of the run into calls, every segment height;
  * default build: the same BITS as the one-step kernel K1a, lattice, av_vels and fields.
K10 runs on a slab that holds the whole grid; the row ny-2 that gets accelerate_flow is
then also the slab's row -2, which the first segment recomputes.
"""
import os

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85


@pytest.fixture
def seg_rows(monkeypatch):
    def set_rows(n):
        monkeypatch.setenv("LBM_TB3_SEG_ROWS", str(n))
    return set_rows


@pytest.mark.parametrize("nx,ny", [(512, 12), (520, 13), (1024, 17), (1540, 12), (2048, 70), (516, 130), (32, 12),
                                   (128, 128), (256, 37), (504, 14), (36, 300)])
@pytest.mark.parametrize("steps", [1, 2, 3, 4, 5, 6, 7, 10])
def test_strict_bit_exact(nx, ny, steps):
    cells, obst = O.random_lattice(nx, ny, seed=nx * 1000 + ny)
    ref, _, av_ref_d = O.run(cells, obst, steps, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_TB3) as lat:
        assert lat.info().kernel == L.KERNEL_TB3
        av = lat.run(steps)
        got = lat.download()
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), \
        "%dx%d: %d cells differ" % (nx, ny, np.count_nonzero((got != ref).any(axis=2)))
    np.testing.assert_allclose(av.astype(np.float64), av_ref_d, rtol=1e-7, atol=0)


@pytest.mark.parametrize("rows_per_segment", [1, 2, 3, 5, 7, 22, 64])
def test_every_segment_height(rows_per_segment, seg_rows):
    seg_rows(rows_per_segment)
    nx, ny, steps = 1024, 23, 6
    cells, obst = O.random_lattice(nx, ny, seed=rows_per_segment, p_obst=0.03)
    ref, _, av_ref_d = O.run(cells, obst, steps, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_TB3) as lat:
        av = lat.run(steps)
        got = lat.download()
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    np.testing.assert_allclose(av.astype(np.float64), av_ref_d, rtol=1e-7, atol=0)


def test_tall_slab_many_segments():
    nx, ny, steps = 1024, 1700, 5
    cells, obst = O.random_lattice(nx, ny, seed=40, p_obst=0.01)
    ref, _, av_ref_d = O.run(cells, obst, steps, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_TB3) as lat:
        av = lat.run(steps)
        _, cs = lat.digest()
    assert cs == L.lattice_checksum(ref)
    np.testing.assert_allclose(av.astype(np.float64), av_ref_d, rtol=1e-7, atol=0)


@pytest.mark.parametrize("nx,ny", [(512, 16), (1024, 40), (2052, 33), (128, 128)])
def test_default_build_gives_the_bits_of_the_one_step_kernel(nx, ny):
    steps = 22
    cells, obst = O.random_lattice(nx, ny, seed=3, p_obst=0.02)
    res = []
    for k in (L.KERNEL_VEC4, L.KERNEL_TB3):
        with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=k) as lat:
            av = lat.run(steps)
            res.append((lat.download(), av, lat.final_fields()))
    assert np.array_equal(res[0][0].view(np.uint32), res[1][0].view(np.uint32))
    assert np.array_equal(res[0][1], res[1][1])
    for a, b in zip(res[0][2], res[1][2]):
        assert np.array_equal(a, b)


def test_long_run_stays_bit_identical_to_the_one_step_kernel():
    """3001 timesteps (1000 three-step passes and a lone step) of a channel with obstacles."""
    nx, ny, steps = 2052, 300, 3001
    cells, obst = O.random_lattice(nx, ny, seed=9, p_obst=0.01)
    res = []
    for k in (L.KERNEL_VEC4, L.KERNEL_TB3):
        with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=k) as lat:
            av = lat.run(steps)
            res.append((lat.digest(), av))
    assert res[0][0] == res[1][0]
    assert np.array_equal(res[0][1], res[1][1]) and np.all(np.isfinite(res[0][1]))


def test_chunked_runs_equal_one_run():
    """run(a); run(b) == run(a+b) with 1-, 2- and 3-step remainders: the K7 and K1a passes
    between K10 passes find the ghost rows K10 pushed."""
    nx, ny = 1024, 24
    cells, obst = O.random_lattice(nx, ny, seed=11)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.KERNEL_TB3) as lat:
        av_all = lat.run(30)
        one = lat.download()
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.KERNEL_TB3) as lat:
        av_parts = np.concatenate([lat.run(n) for n in (1, 3, 0, 5, 2, 1, 4, 7, 3, 2, 2)])
        parts = lat.download()
    assert np.array_equal(one, parts)
    assert np.array_equal(av_all, av_parts)


def test_upload_between_runs():
    nx, ny = 512, 20
    cells, obst = O.random_lattice(nx, ny, seed=21)
    other, _ = O.random_lattice(nx, ny, seed=22)
    ref, _, _ = O.run(other, obst, 6, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | L.KERNEL_TB3) as lat:
        lat.run(4)
        lat.upload(other)
        lat.run(6)
        assert np.array_equal(lat.download(), ref)


def test_selection_and_refusals():
    with L.Lattice(16384, 4096, D, A, W) as lat:
        assert lat.info().kernel == L.KERNEL_TB3                 # beyond L2, enough waves of blocks
    with L.Lattice(4096, 4096, D, A, W) as lat:
        assert lat.info().kernel == L.KERNEL_TB2                 # too few waves: K7
    with L.Lattice(16384, 4096, D, A, W, flags=L.KERNEL_TB2) as lat:
        assert lat.info().kernel == L.KERNEL_TB2                 # forced
    with L.Lattice(16384, 4096, D, A, W, n_gpus=2, device_ids=[0, 0]) as lat:
        assert lat.info().kernel == L.KERNEL_TB2                 # several slabs: K7
    for args in ((130, 64), (512, 11)):
        with pytest.raises(L.LbmError, match="three-step kernel"):
            L.Lattice(*args, D, A, W, flags=L.KERNEL_TB3)
    with pytest.raises(L.LbmError, match="three-step kernel"):
        L.Lattice(512, 40, D, A, W, flags=L.KERNEL_TB3, n_gpus=2, device_ids=[0, 0])
    with pytest.raises(L.LbmError, match="three-step kernel"):
        L.Lattice(512, 40, D, A, W, flags=L.KERNEL_TB3, f64=True)


@pytest.mark.parametrize("steps", [3, 4, 5])
def test_blown_up_lattice_reports_nan(steps):
    nx, ny = 512, 12
    cells, obst = O.random_lattice(nx, ny, seed=2, p_obst=0.0, walls=False)
    cells[4:7, 99:102, :] = 0.0                                  # a hole of zero density: cell (5,100) pulls only zeros, u = 0/0
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.KERNEL_TB3) as lat:
        av = lat.run(steps)
    assert np.isnan(av).all(), av


@settings(max_examples=60, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large],
          derandomize=True)
@given(nxq=st.integers(8, 300), ny=st.integers(12, 40), steps=st.integers(1, 10), seed=st.integers(0, 10 ** 6),
       p_obst=st.sampled_from([0.0, 0.02, 0.2]), density=st.sampled_from([0.1, 0.37]),
       accel=st.sampled_from([0.005, 0.05, 1.1]), omega=st.sampled_from([0.7, 1.0, 1.85]), split=st.integers(0, 10),
       walls=st.booleans(), seg=st.sampled_from([1, 2, 3, 4, 9, 64]))
def test_any_configuration_matches_the_oracle(nxq, ny, steps, seed, p_obst, density, accel, omega, split, walls, seg):
    nx = 4 * nxq
    os.environ["LBM_TB3_SEG_ROWS"] = str(seg)
    try:
        cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=p_obst, walls=walls)
        ref, _, av_ref = O.run(cells, obst, steps, density, accel, omega)
        first = min(split, steps)
        with L.Lattice(nx, ny, density, accel, omega, cells=cells, obstacles=obst,
                       flags=L.STRICT | L.KERNEL_TB3) as lat:
            av = np.concatenate([lat.run(first), lat.run(steps - first)])
            got = lat.download()
            _, cs = lat.digest()
    finally:
        del os.environ["LBM_TB3_SEG_ROWS"]
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert cs == L.lattice_checksum(ref)
    ok = np.isfinite(av_ref)
    assert np.array_equal(np.isfinite(av), ok)
    np.testing.assert_allclose(av[ok].astype(np.float64), av_ref[ok], rtol=1e-6)
