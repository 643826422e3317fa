"""K11 / lbm_gpu_run_batch: many small lattices of one shape advanced together (parameter
sweeps).  Strict build bit-exact against the oracle for every member's own parameters;
default build bit-identical to running the members one after another with lbm_gpu_run,
whatever their history; refusals leave every handle unchanged."""
import ctypes as C

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
PARAMS = [(0.1, 0.005, 1.85), (0.12, 0.004, 1.6), (0.09, 0.006, 1.0), (0.1, 0.003, 1.95), (0.11, 0.005, 1.3)]


def members(nx, ny, b, seed=0, flags=0, p_obst=0.05):
    """b lattices of nx x ny with their own cells, obstacles and (density, accel, omega)."""
    out = []
    for i in range(b):
        cells, obst = O.random_lattice(nx, ny, seed=seed * 1000 + i, p_obst=p_obst)
        d, a, w = PARAMS[i % len(PARAMS)]
        w = w - 0.001 * (i // len(PARAMS))          # every member of a big batch has its own omega
        out.append(dict(cells=cells, obst=obst, prm=(d, a, w), flags=flags))
    return out


def make(m):
    return L.Lattice(m["cells"].shape[1], m["cells"].shape[0], *m["prm"], cells=m["cells"], obstacles=m["obst"],
                     flags=m["flags"])


def state(lat):
    return lat.download(), lat.final_fields(), lat.digest(), lat.info().steps_done


def assert_same(a, b):
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))
    for x, y in zip(a[1], b[1]):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))
    assert a[2] == b[2] and a[3] == b[3]


@pytest.mark.parametrize("nx,ny", [(128, 128), (128, 256), (256, 256), (32, 8), (64, 7), (4, 6), (252, 150), (128, 700)])
@pytest.mark.parametrize("steps", [1, 2, 3, 10])
def test_strict_members_match_the_oracle(nx, ny, steps):
    ms = members(nx, ny, 3, seed=nx + ny, flags=L.STRICT | L.KERNEL_PAIRS)
    lats = [make(m) for m in ms]
    assert all(lat.info().kernel == L.KERNEL_PAIRS for lat in lats)
    av = L.run_batch(lats, steps)
    assert av.shape == (3, steps) and av.dtype == np.float32
    for m, lat, row in zip(ms, lats, av):
        ref, _, av_ref = O.run(m["cells"], m["obst"], steps, *m["prm"])
        got = lat.download()
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), \
            "%dx%d: %d cells differ" % (nx, ny, np.count_nonzero((got != ref).any(axis=2)))
        np.testing.assert_allclose(row.astype(np.float64), av_ref, rtol=1e-7, atol=0)
        assert lat.info().steps_done == steps
        lat.close()


@pytest.mark.parametrize("b,steps", [(1, 9), (2, 10), (7, 33), (120, 11)])
def test_default_build_equals_solo_runs(b, steps):
    ms = members(128, 128, b, seed=b)
    batch = [make(m) for m in ms]
    solo = [make(m) for m in ms]
    av = L.run_batch(batch, steps)
    for i, (x, y) in enumerate(zip(batch, solo)):
        av_solo = y.run(steps)
        assert np.array_equal(av[i].view(np.uint32), av_solo.view(np.uint32)), i
        assert_same(state(x), state(y))
        assert x.info().last_run_device_ms == batch[0].info().last_run_device_ms
    for lat in batch + solo:
        lat.close()


@pytest.mark.parametrize("a,b", [(3, 4), (4, 5), (2, 2), (1, 1)])
def test_mixed_histories(a, b):
    nx, ny = 128, 96
    ms = members(nx, ny, 3, seed=7)
    batch = [make(m) for m in ms]
    solo = [make(m) for m in ms]
    fresh_cells, _ = O.random_lattice(nx, ny, seed=99)
    for group in (batch, solo):
        group[0].run(3)                       # other buffer parity, steps_done = 3
        group[1].run(2)
        group[1].upload(fresh_cells)          # just uploaded
    av1 = L.run_batch(batch, a)
    av2 = L.run_batch(batch, b)
    for i, (x, y) in enumerate(zip(batch, solo)):
        s1, s2 = y.run(a), y.run(b)
        assert np.array_equal(av1[i].view(np.uint32), s1.view(np.uint32)), i
        assert np.array_equal(av2[i].view(np.uint32), s2.view(np.uint32)), i
        assert_same(state(x), state(y))
    # a solo run continues from where the batch left the member
    assert np.array_equal(batch[0].run(5).view(np.uint32), solo[0].run(5).view(np.uint32))
    assert_same(state(batch[0]), state(solo[0]))
    for lat in batch + solo:
        lat.close()


def test_run_longer_than_one_segment():
    steps = 65537                                 # > kMaxSegmentSteps (1 << 16), odd
    ms = members(32, 8, 3, seed=11)
    batch = [make(m) for m in ms]
    av = L.run_batch(batch, steps)
    for i, (m, x) in enumerate(zip(ms, batch)):
        with make(m) as y:
            av_solo = y.run(steps)
            assert np.array_equal(av[i].view(np.uint32), av_solo.view(np.uint32)), i
            assert_same(state(x), state(y))
        x.close()


def test_nan_stays_in_its_own_row():
    nx, ny = 64, 12
    ms = members(nx, ny, 3, seed=2, p_obst=0.0)
    ms[1]["cells"] = ms[1]["cells"].copy()
    ms[1]["cells"][4:7, 19:22, :] = 0.0           # blows up (density 0 -> division by zero)
    batch = [make(m) for m in ms]
    av = L.run_batch(batch, 4)
    assert np.isnan(av[1]).all(), av[1]
    for i in (0, 2):
        assert np.isfinite(av[i]).all()
        with make(ms[i]) as y:
            assert np.array_equal(av[i].view(np.uint32), y.run(4).view(np.uint32))
            assert_same(state(batch[i]), state(y))
    for lat in batch:
        lat.close()


def _raw(handles, n, steps):
    lib = L.load_library()
    arr = (C.c_void_p * max(len(handles), 1))(*handles)
    rc = lib.lbm_gpu_run_batch(C.cast(arr, C.c_void_p), n, steps, None)
    return rc, lib.lbm_gpu_last_error().decode()


def test_refusals_change_nothing():
    D, A, W = 0.1, 0.005, 1.85
    a = L.Lattice(128, 128, D, A, W)
    b = L.Lattice(128, 128, D, A, W)
    a.run(3)
    others = {
        "same nx and ny": [L.Lattice(128, 64, D, A, W), L.Lattice(64, 128, D, A, W)],
        "STRICT": [L.Lattice(128, 128, D, A, W, flags=L.STRICT)],
        "double precision": [L.Lattice(128, 128, D, A, W, f64=True)],
        "pairs kernel": [L.Lattice(512, 512, D, A, W), L.Lattice(128, 128, D, A, W, flags=L.KERNEL_VEC4)],
        "slabs": [L.Lattice(128, 128, D, A, W, n_gpus=2, device_ids=[0, 0])],
    }
    before = [(lat, lat.digest(), lat.info().steps_done) for lat in [a, b] + sum(others.values(), [])]
    for what, lats in others.items():
        for o in lats:
            rc, msg = _raw([a.h.value, o.h.value, b.h.value], 3, 4)
            assert rc != 0 and msg.startswith("lbm_gpu_run_batch:") and what in msg, msg
    rc, msg = _raw([a.h.value, b.h.value, a.h.value], 3, 4)
    assert rc != 0 and msg.startswith("lbm_gpu_run_batch:") and "duplicate" in msg, msg
    rc, msg = _raw([a.h.value, None], 2, 4)
    assert rc != 0 and msg.startswith("lbm_gpu_run_batch:") and "NULL" in msg, msg
    rc, msg = _raw([a.h.value], 0, 4)
    assert rc != 0 and msg.startswith("lbm_gpu_run_batch:") and "at least one" in msg, msg
    rc, msg = _raw([a.h.value, b.h.value], 2, -1)
    assert rc != 0 and msg.startswith("lbm_gpu_run_batch:") and "negative" in msg, msg
    with pytest.raises(L.LbmError, match="lbm_gpu_run_batch: .*same nx and ny"):
        L.run_batch([a, others["same nx and ny"][0]], 2)
    for lat, dig, steps in before:
        assert lat.digest() == dig and lat.info().steps_done == steps
    for lat in [a, b] + sum(others.values(), []):
        lat.close()


def test_refuses_members_on_different_devices():
    if L.load_library().lbm_gpu_device_count() < 2:
        pytest.skip("needs two GPUs")
    a = L.Lattice(128, 128, 0.1, 0.005, 1.85, device_ids=[0])
    b = L.Lattice(128, 128, 0.1, 0.005, 1.85, device_ids=[1])
    rc, msg = _raw([a.h.value, b.h.value], 2, 4)
    assert rc != 0 and "device" in msg, msg
    a.close()
    b.close()


@settings(max_examples=25, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large])
@given(nx4=st.integers(1, 64), ny=st.integers(4, 300), b=st.integers(1, 6), steps=st.integers(0, 12),
       seed=st.integers(0, 10 ** 6))
def test_property_batch_equals_solo(nx4, ny, b, steps, seed):
    nx = 4 * nx4
    ms = members(nx, ny, b, seed=seed)
    batch = [make(m) for m in ms]
    if any(lat.info().kernel != L.KERNEL_PAIRS for lat in batch):      # e.g. large grids go elsewhere
        for lat in batch:
            lat.close()
        return
    av = L.run_batch(batch, steps)
    for i, (m, x) in enumerate(zip(ms, batch)):
        with make(m) as y:
            assert np.array_equal(av[i].view(np.uint32), y.run(steps).view(np.uint32)), i
            assert_same(state(x), state(y))
        x.close()
