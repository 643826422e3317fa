"""LBM_GPU_STORE_F16: the lattice stored as shifted binary16 (f_k - c_k, c_k the rest state),
the arithmetic in fp32.  K1a-f16 does one step per pass, K7-f16 two.

  * strict build: bit-exact against oracle_f16.run_f16 (the fp32 oracle one step at a time,
    encoded and decoded with numpy between steps), lattice and av_vels;
  * default build: K7-f16 gives the bits of K1a-f16, and any split of a run gives the bits
    of the whole run;
  * the handle reads back decoded fp32 values, and writes encoded ones;
  * what the flag does not support is refused without touching any handle.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import lbm_b200 as L
import oracle_f16 as H
import oracle_lib as O
import readout_ref as R

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85
F16 = L.STORE_F16
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def k7_applies(nx, ny):
    """K7-f16 runs by default where K7's shape rules hold and nx is a multiple of 8."""
    return nx % 8 == 0 and nx >= 32 and ny >= 8


def bits_equal(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


@pytest.mark.parametrize("nx,ny", [(128, 128), (128, 256), (256, 256), (4, 6), (32, 8), (64, 7), (130, 20),
                                   (252, 150), (1024, 24)])
@pytest.mark.parametrize("steps", [1, 2, 3, 10])
@pytest.mark.parametrize("forced", [L.KERNEL_VEC4, 0])
def test_strict_bit_exact_against_the_oracle(nx, ny, steps, forced):
    cells, obst = O.random_lattice(nx, ny, seed=nx * 1000 + ny)
    ref, av_ref = H.run_f16(cells, obst, steps, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.STRICT | F16 | forced) as lat:
        assert lat.info().kernel == (L.KERNEL_TB2 if not forced and k7_applies(nx, ny) else L.KERNEL_VEC4)
        av = lat.run(steps)
        got = lat.download()
    assert bits_equal(got, ref), "%dx%d: %d cells differ" % (nx, ny, np.count_nonzero((got != ref).any(axis=2)))
    np.testing.assert_allclose(av.astype(np.float64), av_ref, rtol=1e-7, atol=0)


def test_k7_f16_equals_k1a_f16_over_1001_steps():
    nx, ny, steps = 1032, 300, 1001
    cells, obst = O.random_lattice(nx, ny, seed=9, p_obst=0.01)
    res = []
    for k in (L.KERNEL_VEC4, 0):
        with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=F16 | k) as lat:
            av = lat.run(steps)
            res.append((lat.info().kernel, lat.digest(), av, lat.final_fields()))
    assert (res[0][0], res[1][0]) == (L.KERNEL_VEC4, L.KERNEL_TB2)
    assert res[0][1] == res[1][1]
    assert np.array_equal(res[0][2], res[1][2]) and np.all(np.isfinite(res[0][2]))
    for a, b in zip(res[0][3], res[1][3]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("first", [3, 4])
def test_split_run_equals_one_run(first):
    nx, ny, steps = 512, 40, 13
    cells, obst = O.random_lattice(nx, ny, seed=11)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=F16) as lat:
        av_all = lat.run(steps)
        one = lat.download()
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=F16) as lat:
        av_parts = np.concatenate([lat.run(first), lat.run(steps - first)])
        parts = lat.download()
    assert bits_equal(one, parts)
    assert np.array_equal(av_all, av_parts)


@pytest.mark.parametrize("nx,ny", [(256, 64), (252, 40)])
def test_default_build_close_to_the_oracle(nx, ny):
    """The default arithmetic differs from the reference order by a few fp32 roundings per cell
    and step.  After the encode that either vanishes or moves a stored value by one binary16
    step, so the lattice may drift from the strict result by about one binary16 ulp of the
    largest stored value per step: the bound is steps x that ulp.  av_vels averages |u| over
    all cells, where a few such cells change it by far less than 1e-4 relative."""
    steps = 50
    cells, obst = O.random_lattice(nx, ny, seed=5, p_obst=0.02)
    ref, av_ref = H.run_f16(cells, obst, steps, D, A, W)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=F16) as lat:
        av = lat.run(steps)
        got = lat.download()
    ulp = float(np.spacing(np.abs(H.f16_encode(ref, D)).max()))
    assert np.abs(got.astype(np.float64) - ref).max() <= steps * ulp
    np.testing.assert_allclose(av.astype(np.float64), av_ref, rtol=1e-4)


def test_fresh_lattice_is_the_exact_rest_state():
    nx, ny = 96, 20
    with L.Lattice(nx, ny, D, A, W, flags=F16) as lat:
        assert bits_equal(lat.download(), O.rest_cells(nx, ny, D))
        assert lat.digest()[1] == L.lattice_checksum(O.rest_cells(nx, ny, D))


@pytest.mark.parametrize("nx,ny", [(128, 32), (130, 9)])
def test_upload_and_create_encode_as_numpy_does(nx, ny):
    cells, obst = O.random_lattice(nx, ny, seed=3)
    want = H.f16_decode(H.f16_encode(cells, D), D)
    with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=F16) as lat:
        assert bits_equal(lat.download(), want)
        lat.run(3)
        lat.upload(cells)
        got = lat.download()
        assert bits_equal(got, want)
        assert bits_equal(lat.download_rows(2, 5), want[2:7])
        mass, cs = lat.digest()
        assert cs == L.lattice_checksum(got)
        assert mass == pytest.approx(float(np.sum(got.astype(np.float64))), rel=1e-7)
        ux, uy, u, p = lat.final_fields()
        rux, ruy, ru, rp = O.final_state(want, obst, np.float32(D))
        assert bits_equal(u, ru) and bits_equal(p, rp)
        _, tot, n = O.av_velocity(want, obst)          # the oracle's double sum: the device sum is exact
        assert lat.av_velocity() == pytest.approx(tot / n, rel=1e-6)
        assert lat.av_velocity() == R.host_average(R.fixed_u_sum(ru, obst), n, np.float32)
        assert mass == R.digest_mass(got)


def test_device_bytes_show_the_saving():
    nx, ny = 8192, 4096
    with L.Lattice(nx, ny, D, A, W) as lat:
        full = lat.info().device_bytes
    with L.Lattice(nx, ny, D, A, W, flags=F16) as lat:
        half = lat.info().device_bytes
        assert lat.info().kernel == L.KERNEL_TB2
    assert half <= 0.55 * full, (half, full)


@pytest.mark.parametrize("forced", [L.KERNEL_VEC4, 0])
def test_nan_is_reported_as_for_fp32(forced):
    nx, ny, steps = 512, 24, 3
    cells, obst = O.random_lattice(nx, ny, seed=2, p_obst=0.0, walls=False)
    cells[10, 100, :] = np.nan
    avs = []
    for flags in (forced, F16 | forced):
        with L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=flags) as lat:
            avs.append(lat.run(steps))
    assert np.isnan(avs[0]).all() and np.isnan(avs[1]).all(), avs


def test_refusals_leave_every_handle_unchanged():
    nx, ny = 64, 32
    with L.Lattice(nx, ny, D, A, W, flags=F16) as lat, L.Lattice(nx, ny, D, A, W) as other:
        lat.run(3)
        other.run(2)
        assert other.info().kernel == L.KERNEL_PAIRS

        def state():
            return [(h.digest(), h.info().steps_done) for h in (lat, other)]

        before = state()
        refused = [(dict(f64=True), "fp32 lattices only"),
                   (dict(n_gpus=2, device_ids=[0, 0]), "n_gpus == 1"),
                   (dict(slab=(0, ny)), "not slab handles")]
        for k in (L.KERNEL_SCALAR, L.KERNEL_TMA, L.KERNEL_PERSISTENT, L.KERNEL_CLUSTER, L.KERNEL_PAIRS, L.KERNEL_TB3):
            refused.append((dict(flags=F16 | k), "VEC4 or LBM_GPU_KERNEL_TB2 only"))
        for kw, msg in refused:
            kw.setdefault("flags", F16)
            with pytest.raises(L.LbmError, match=msg):
                L.Lattice(nx, ny, D, A, W, **kw)
        with pytest.raises(L.LbmError, match="multiple of 8"):
            L.Lattice(68, ny, D, A, W, flags=F16 | L.KERNEL_TB2)
        with pytest.raises(L.LbmError, match="pairs kernel"):
            L.run_batch([other, lat], 4)
        with pytest.raises(L.LbmError, match="shared between processes"):
            lat.ipc_export()
        assert state() == before


@settings(max_examples=50, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large],
          derandomize=True)
@given(nx=st.integers(1, 600), ny=st.integers(2, 40), steps=st.integers(1, 9), seed=st.integers(0, 10 ** 6),
       p_obst=st.sampled_from([0.0, 0.02, 0.2]), density=st.sampled_from([0.1, 0.37]),
       accel=st.sampled_from([0.005, 0.05]), omega=st.sampled_from([0.7, 1.0, 1.85]), split=st.integers(0, 9),
       walls=st.booleans(), forced=st.sampled_from([0, L.KERNEL_VEC4]))
def test_any_configuration_matches_the_oracle(nx, ny, steps, seed, p_obst, density, accel, omega, split, walls, forced):
    cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=p_obst, walls=walls)
    ref, av_ref = H.run_f16(cells, obst, steps, density, accel, omega)
    first = min(split, steps)
    with L.Lattice(nx, ny, density, accel, omega, cells=cells, obstacles=obst, flags=L.STRICT | F16 | forced) as lat:
        av = np.concatenate([lat.run(first), lat.run(steps - first)])
        got = lat.download()
        _, cs = lat.digest()
    assert bits_equal(got, ref)
    assert cs == L.lattice_checksum(ref)
    ok = np.isfinite(av_ref)
    assert np.array_equal(np.isfinite(av), ok)
    np.testing.assert_allclose(av[ok].astype(np.float64), av_ref[ok], rtol=1e-6)


@pytest.mark.parametrize("name", ["128x128", "128x256"])
def test_cli_f16_passes_check(name, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import expand_golden
    expand_golden.expand(name, str(tmp_path))
    env = dict(os.environ, LBM_PRECISION="f16")
    r = subprocess.run([os.path.join(ROOT, "d2q9-bgk"), os.path.join(ROOT, "inputs", "input_%s.params" % name),
                        os.path.join(ROOT, "inputs", "obstacles_%s.dat" % name)],
                       cwd=str(tmp_path), env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([sys.executable, os.path.join(ROOT, "check", "check.py"),
                        "--ref-av-vels-file=" + os.path.join(str(tmp_path), name + ".av_vels.dat"),
                        "--ref-final-state-file=" + os.path.join(str(tmp_path), name + ".final_state.dat"),
                        "--av-vels-file=" + os.path.join(str(tmp_path), "av_vels.dat"),
                        "--final-state-file=" + os.path.join(str(tmp_path), "final_state.dat")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
