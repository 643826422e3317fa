"""The default build (what ./d2q9-bgk, bench.py and every kernel without LBM_GPU_STRICT run):

  1. every default kernel of one precision gives the bits of K1a on one slab: the lattice,
     the exact per-step |u| sums (run_sums) and final_fields, for any small grid, mask,
     parameters, slab count, tuning knob and split of the run into calls;
  2. each step of K1a (fp32 and fp64) stays within default_ref.bound() of the same step in
     extended precision, taken from the GPU's own previous state; part 1 carries this to
     every other kernel and to the multi-step passes;
  3. one |u| limit: a step in which one fluid cell reaches |u| >= 2 reads NaN in every kernel
     and both builds, whichever cell of its quad it is, and av_velocity() agrees with run().
"""
import contextlib
import os

import numpy as np
import pytest
from hypothesis import HealthCheck, given, settings, strategies as st

import default_ref as R
import lbm_b200 as L
import oracle_lib as O
import readout_ref as RR

pytestmark = pytest.mark.gpu

OMEGAS = [0.5, 1.0, 1.5, 1.85, 1.99]
DENSITIES = [0.01, 0.1, 1.0]
ACCELS = [0.005, 1.1]          # 1.1 turns the accelerate_flow guard false on part of row ny-2


@contextlib.contextmanager
def env(**knobs):
    """Tuning knobs are read when a lattice is created."""
    old = {k: os.environ.get(k) for k in knobs}
    os.environ.update({k: str(v) for k, v in knobs.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def lattice(cells, obst, prm, flags, n=1, f64=False, **knobs):
    ny, nx, _ = cells.shape
    with env(**knobs):
        return L.Lattice(nx, ny, *prm, cells=cells, obstacles=obst, flags=flags, n_gpus=n, device_ids=[0] * n,
                         f64=f64)


def fits(cells, obst, prm, flags, n=1, f64=False, **knobs):
    """The lattice, or None where the kernel refuses this shape."""
    try:
        return lattice(cells, obst, prm, flags, n, f64, **knobs)
    except L.LbmError:
        return None


def outcome(lat, first, steps):
    """(lattice, per-step sums, final_fields) after run_sums over a run split into two calls."""
    sums = np.concatenate([lat.run_sums(first), lat.run_sums(steps - first)])
    out = (lat.download(), sums, lat.final_fields())
    lat.close()
    return out


def assert_same_bits(got, want, what):
    cells, sums, fields = got
    assert np.array_equal(cells.view(np.uint8), want[0].view(np.uint8)), \
        "%s: %d cells differ" % (what, np.count_nonzero((cells != want[0]).any(axis=2)))
    assert np.array_equal(sums.view(np.uint64), want[1].view(np.uint64)), "%s: sums %s != %s" % (what, sums, want[1])
    for a, b in zip(fields, want[2]):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), what


# ------------------------------------------------------------------ 1. same bits
@settings(max_examples=120, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large],
          derandomize=True)
@given(nx=st.integers(1, 300), ny=st.integers(2, 40), steps=st.integers(1, 7), seed=st.integers(0, 10 ** 6),
       p_obst=st.sampled_from([0.0, 0.02, 0.2, 0.6]), walls=st.booleans(), slabs=st.integers(1, 4),
       density=st.sampled_from(DENSITIES), accel=st.sampled_from(ACCELS), omega=st.sampled_from(OMEGAS),
       split=st.integers(0, 7), members=st.integers(1, 3), seg=st.sampled_from([2, 3, 5, 9, 64]),
       tail=st.sampled_from([0, 2, 4]))
def test_every_default_kernel_gives_the_bits_of_k1a(nx, ny, steps, seed, p_obst, walls, slabs, density, accel,
                                                    omega, split, members, seg, tail):
    prm = (density, accel, omega)
    cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=p_obst, walls=walls)
    first = min(split, steps)
    base = outcome(lattice(cells, obst, prm, L.KERNEL_VEC4), first, steps)
    n = min(slabs, ny)
    runs = {
        "K1b": lattice(cells, obst, prm, L.KERNEL_SCALAR),
        "K1c": lattice(cells, obst, prm, L.KERNEL_TMA),
        "K5": lattice(cells, obst, prm, L.KERNEL_PERSISTENT),
        "K5 scalar tiles": lattice(cells, obst, prm, L.KERNEL_PERSISTENT, LBM_PERSIST_VEC=1),
        "K1a %d slabs" % n: lattice(cells, obst, prm, L.KERNEL_VEC4, n),
        "K1b %d slabs" % n: lattice(cells, obst, prm, L.KERNEL_SCALAR, n),
        "K6": fits(cells, obst, prm, L.KERNEL_CLUSTER),
        "K9": fits(cells, obst, prm, L.KERNEL_PAIRS),
        "K7": fits(cells, obst, prm, L.KERNEL_TB2, LBM_TB2_SEG_ROWS=seg, LBM_TB2_TAIL_ROWS=tail),
        "K7 %d slabs" % n: fits(cells, obst, prm, L.KERNEL_TB2, n if ny // n >= 8 else 1, LBM_TB2_SEG_ROWS=seg),
        "K10": fits(cells, obst, prm, L.KERNEL_TB3, LBM_TB3_SEG_ROWS=seg),
    }
    if nx % 4 == 0 and nx <= 256 and ny >= 4:
        assert runs["K9"] is not None, "K9 refused a shape it runs"
    if nx % 4 == 0 and nx >= 32 and ny >= 8:
        assert runs["K7"] is not None, "K7 refused a shape it runs"
    for name, lat in runs.items():
        if lat is not None:
            assert_same_bits(outcome(lat, first, steps), base, name)

    # K11: the members of one batch, each with the bits of its solo K1a run
    if runs["K9"] is not None:
        ms = [(cells if i == 0 else O.random_lattice(nx, ny, seed=seed + i, density=density, p_obst=p_obst,
                                                    walls=walls)[0]) for i in range(members)]
        batch = [lattice(c, obst, prm, L.KERNEL_PAIRS) for c in ms]
        av = np.concatenate([L.run_batch(batch, k) for k in (first, steps - first) if k > 0], axis=1)
        for i, (c, lat) in enumerate(zip(ms, batch)):
            with lattice(c, obst, prm, L.KERNEL_VEC4) as solo:
                want = solo.run(steps)
                want_cells, want_fields = solo.download(), solo.final_fields()
            assert np.array_equal(av[i].view(np.uint32), want.view(np.uint32)), "K11 member %d" % i
            assert np.array_equal(lat.download().view(np.uint32), want_cells.view(np.uint32)), "K11 member %d" % i
            for a, b in zip(lat.final_fields(), want_fields):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), "K11 member %d" % i
            lat.close()

    # binary16 storage: K7-f16 against K1a-f16
    if nx % 8 == 0 and nx >= 32 and ny >= 8:
        f16 = outcome(lattice(cells, obst, prm, L.STORE_F16 | L.KERNEL_VEC4), first, steps)
        assert_same_bits(outcome(lattice(cells, obst, prm, L.STORE_F16 | L.KERNEL_TB2, LBM_TB2_SEG_ROWS=seg),
                                 first, steps), f16, "K7-f16")


@settings(max_examples=40, deadline=None, suppress_health_check=[HealthCheck.too_slow, HealthCheck.data_too_large],
          derandomize=True)
@given(nx=st.integers(1, 300), ny=st.integers(3, 40), steps=st.integers(1, 7), seed=st.integers(0, 10 ** 6),
       p_obst=st.sampled_from([0.0, 0.02, 0.2, 0.6]), walls=st.booleans(), density=st.sampled_from(DENSITIES),
       accel=st.sampled_from(ACCELS), omega=st.sampled_from(OMEGAS), split=st.integers(0, 7))
def test_fp64_default_kernels_give_the_same_bits(nx, ny, steps, seed, p_obst, walls, density, accel, omega, split):
    prm = (density, accel, omega)
    cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=p_obst, walls=walls,
                                   dtype=np.float64)
    first = min(split, steps)

    def run(flags, n=1):
        lat = lattice(cells, obst, prm, flags, n, f64=True)
        av = np.concatenate([lat.run(first), lat.run(steps - first)])
        out = (lat.download(), av, lat.final_fields())
        lat.close()
        return out

    base = run(L.KERNEL_SCALAR)
    for name, got in [("K1a", run(L.KERNEL_VEC4)), ("K1a 3 slabs", run(L.KERNEL_VEC4, 3)),
                      ("K1b 3 slabs", run(L.KERNEL_SCALAR, 3)), ("K5", run(L.KERNEL_PERSISTENT))]:
        assert_same_bits(got, base, name)


# ------------------------------------------------------------------ 2. within the bound
def bound_lattices(nx, ny, density, seed, dtype):
    """A random lattice, and one with negative speeds (a third of the values moved by up to
    -15 % / +15 % of the density)."""
    cells, obst = O.random_lattice(nx, ny, seed=seed, density=density, p_obst=0.05, dtype=dtype)
    rng = np.random.default_rng(seed)
    neg = cells.copy()
    pick = rng.random(neg.shape) < 1 / 3
    neg[pick] += (density * rng.uniform(-0.15, 0.15, int(pick.sum()))).astype(dtype)
    assert (neg < 0).any()
    return [("random", cells, obst), ("negative speeds", neg, obst)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("accel", ACCELS)
@pytest.mark.parametrize("density", DENSITIES)
def test_each_step_is_within_the_bound_of_the_exact_step(dtype, accel, density):
    nx, ny, steps = 70, 14, 5
    eps = R.eps_of(dtype)
    worst = 0.0
    for omega in OMEGAS:
        for name, cells, obst in bound_lattices(nx, ny, density, 17, dtype):
            with lattice(cells, obst, (density, accel, omega), L.KERNEL_VEC4, f64=dtype == np.float64) as lat:
                prev = cells
                for t in range(steps):
                    av = lat.run(1)[0]
                    got = lat.download()
                    ref = R.f64_step(prev, obst, density, accel, omega)
                    b, bu = R.bound(ref["pulled"], ref["omega"], eps, obst=obst)
                    err = np.abs(got.astype(np.longdouble) - ref["cells"]).astype(np.float64)
                    where = "%s, omega %s, step %d" % (name, omega, t + 1)
                    assert (err <= b).all(), "%s: %d values beyond the bound, worst ratio %.3g" % (
                        where, np.count_nonzero(err > b), np.max(err / np.where(b > 0, b, 1)))
                    fluid = obst == 0
                    speed = ref["speed"][fluid].astype(np.float64)
                    if np.all(speed + bu[fluid] < RR.SPEED_LIMIT):
                        exact_av = float(np.sum(ref["speed"][fluid], dtype=np.longdouble) / fluid.sum())
                        tol = R.av_bound(ref["speed"], bu, obst, eps)
                        assert abs(float(av) - exact_av) <= tol, "%s: av_vels %r, exact %r" % (where, av, exact_av)
                    elif np.any(speed - bu[fluid] >= RR.SPEED_LIMIT):     # a cell surely beyond the limit
                        assert np.isnan(av), "%s: av_vels %r with |u| up to %r" % (where, av, speed.max())
                    worst = max(worst, float(np.max(err[fluid] / b[fluid])))
                    prev = got
    print("largest error / bound on the GPU: %.3f" % worst)


# ------------------------------------------------------------------ 3. one |u| limit
NX, NY, D, A, W = 64, 12, 0.1, 0.005, 1.85


def blow_up(nx=NX, ny=NY, x=22, y=5):
    """Cell (x, y) pulls p1 = 0.5 from the west, p3 = -0.3 from the east and zeros otherwise:
    rho 0.2 and |u| ~ 4 after one step, while every other cell stays far below the limit and
    its quad's |u| sum below 8 (the quad bound the default build used to apply)."""
    cells, obst = O.random_lattice(nx, ny, seed=3, p_obst=0.0, walls=False)
    obst[:] = 0
    for k in range(9):
        cells[(y - R.CY[k]) % ny, (x - R.CX[k]) % nx, k] = 0.0
    cells[y, (x - 1) % nx, 1], cells[y, (x + 1) % nx, 3] = 0.5, -0.3
    return cells, obst


def strict_speeds(cells, obst, steps):
    """|u| of every cell at each step of the strict oracle run."""
    out, c = [], cells
    for _ in range(steps):
        c, sp = RR.strict_step_speeds(c, obst, D, A, W)
        out.append(sp)
    return out


def assert_clear_crossing(cells, obst, step):
    """The oracle's first |u| >= 2 is at `step` (1-based), in cells whose quad sums stay below 8,
    and no cell up to that step is within 1e-3 of the limit (so both builds agree)."""
    sp = strict_speeds(cells, obst, step)
    for t, s in enumerate(sp):
        assert np.isfinite(s).all()
        assert np.min(np.abs(s - RR.SPEED_LIMIT)) > 1e-3
        quads = np.pad(s, ((0, 0), (0, (-s.shape[1]) % 4))).reshape(s.shape[0], -1, 4).sum(axis=-1)
        assert quads.max() < 8.0
        assert (s.max() >= RR.SPEED_LIMIT) == (t == step - 1)


def kernels_for(nx, ny, slabs):
    """(name, flags, n_slabs) of every fp32 kernel that runs this shape."""
    out = [("K1a", L.KERNEL_VEC4, 1), ("K1b", L.KERNEL_SCALAR, 1), ("K1c", L.KERNEL_TMA, 1),
           ("K5", L.KERNEL_PERSISTENT, 1), ("K6", L.KERNEL_CLUSTER, 1)]
    if slabs > 1:
        out += [("K1a %d slabs" % slabs, L.KERNEL_VEC4, slabs), ("K1b %d slabs" % slabs, L.KERNEL_SCALAR, slabs)]
    if nx % 4 == 0 and nx <= 256:
        out.append(("K9", L.KERNEL_PAIRS, 1))
    if nx % 4 == 0 and nx >= 32:
        out.append(("K7", L.KERNEL_TB2, 1))
        if ny // slabs >= 8 and slabs > 1:
            out.append(("K7 %d slabs" % slabs, L.KERNEL_TB2, slabs))
        if ny >= 12:
            out.append(("K10", L.KERNEL_TB3, 1))
    if nx % 8 == 0 and nx >= 32:
        out += [("K1a-f16", L.STORE_F16 | L.KERNEL_VEC4, 1), ("K7-f16", L.STORE_F16 | L.KERNEL_TB2, 1)]
    return out


def check_every_kernel(cells, obst, steps, slabs=1):
    ny, nx, _ = cells.shape
    want = {f16: RR.strict_av_vels(cells, obst, steps, D, A, W, f16=f16)[1] for f16 in (False, True)}
    for name, flags, n in kernels_for(nx, ny, slabs):
        exp = want[bool(flags & L.STORE_F16)]
        for build, strict in (("default", 0), ("strict", L.STRICT)):
            with lattice(cells, obst, (D, A, W), flags | strict, n) as lat:
                av = lat.run(steps)
                readout = lat.av_velocity()
            what = "%s, %s build" % (name, build)
            assert np.array_equal(np.isnan(av), np.isnan(exp)), "%s: %s, expected %s" % (what, av, exp)
            assert np.isnan(readout) == np.isnan(av[-1]), "%s: av_velocity %r after %s" % (what, readout, av)


@pytest.mark.parametrize("x,y,nx,slabs", [
    (20, 5, NX, 1), (21, 5, NX, 1), (22, 5, NX, 1), (23, 5, NX, 1),     # x mod 4 = 0, 1, 2, 3
    (64, 5, 66, 1), (65, 5, 66, 1),                                      # the ragged last quad
    (22, 5, NX, 2), (22, 6, NX, 2),                                      # either side of a slab boundary
    (22, NY - 2, NX, 1),                                                 # the accelerated row
])
def test_one_fast_cell_makes_the_step_nan_in_every_kernel(x, y, nx, slabs):
    cells, obst = blow_up(nx=nx, x=x, y=y)
    assert_clear_crossing(cells, obst, 1)
    check_every_kernel(cells, obst, 1, slabs)
    obst[y, x] = 1                            # the same cell as an obstacle: nothing to report
    assert np.isfinite(RR.strict_av_vels(cells, obst, 1, D, A, W)[1]).all()
    check_every_kernel(cells, obst, 1, slabs)


@pytest.mark.parametrize("seed,step", [(0, 2), (3402, 3)])
def test_the_later_steps_of_a_pass_mark_their_own_step(seed, step):
    """K7 and K10 advance two and three steps per pass: a crossing at the second or third step
    must make that step NaN, not the pass's first."""
    cells, obst = O.random_lattice(NX, NY, seed=3, p_obst=0.0, walls=False)
    obst[:] = 0
    rng = np.random.default_rng(seed)
    blk = cells[3:8, 19:26]
    blk[:] = (rng.uniform(-0.02, 0.05, blk.shape).astype(np.float32) *
              rng.uniform(0, 1, blk.shape[:2])[..., None].astype(np.float32))
    assert_clear_crossing(cells, obst, step)
    check_every_kernel(cells, obst, step)


def test_k11_member_nan_stays_in_its_row():
    cells, obst = blow_up()
    calm, _ = O.random_lattice(NX, NY, seed=4, p_obst=0.0, walls=False)
    for strict in (0, L.STRICT):
        batch = [lattice(c, obst, (D, A, W), L.KERNEL_PAIRS | strict) for c in (calm, cells, calm)]
        av = L.run_batch(batch, 1)
        assert np.isnan(av[1, 0]) and np.isfinite(av[[0, 2], 0]).all(), av
        assert np.isnan(batch[1].av_velocity())
        for lat in batch:
            lat.close()
