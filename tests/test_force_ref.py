"""tests/force_ref.py against the header's formula evaluated term by term in fractions.Fraction,
and the momentum balance P_fluid(t+1) = P~_fluid(t) - F_all(t) on the oracle's own step.  CPU only."""
import math
from fractions import Fraction

import numpy as np
import pytest

import force_ref as F
import oracle_lib as O


def formula(tilde, obst, boxes):
    """F_B(t) of include/lbm_gpu.h, literally: per solid cell in B, the momentum streaming in from
    fluid neighbours minus the momentum it sends to them, each value rounded to 2^-32 half to even
    (Python's round of a Fraction), the sum converted to the nearest double."""
    ny, nx, _ = tilde.shape
    out = []
    for (x0, y0, x1, y1) in boxes:
        sx = sy = Fraction(0)
        bad = False
        for y in range(y0, y1):
            for x in range(x0, x1):
                if not obst[y, x]:
                    continue
                for k in range(1, 9):
                    cx, cy = F.CK[k]
                    terms = []
                    if not obst[(y - cy) % ny, (x - cx) % nx]:
                        terms.append((1, tilde[(y - cy) % ny, (x - cx) % nx, k]))
                    if not obst[(y + cy) % ny, (x + cx) % nx]:
                        terms.append((-1, tilde[y, x, k]))
                    for sign, v in terms:
                        if not abs(float(v)) < 2.0 ** 31:
                            bad = True
                            continue
                        q = round(Fraction(float(v)) * 2 ** 32)
                        sx += sign * cx * q
                        sy += sign * cy * q
        out.append((math.nan, math.nan) if bad else (float(sx / 2 ** 32), float(sy / 2 ** 32)))
    return np.array(out, dtype=np.float64)


def small_case(nx, ny, seed, dtype):
    rng = np.random.default_rng(seed)
    cells, obst = O.random_lattice(nx, ny, seed, p_obst=0.3, dtype=dtype)
    obst[:, 0] |= rng.random(ny) < 0.5                     # obstacles on both wrap edges
    obst[:, nx - 1] |= rng.random(ny) < 0.5
    obst[ny - 1, rng.integers(0, nx)] = 1
    # ties at 2^-33 (v * 2^32 = n + 1/2), tiny values, and negatives
    cells[..., 1] += dtype(3 * 2.0 ** -33)
    cells[0, 0, 5] = dtype(-5 * 2.0 ** -33)
    cells[1, 1, 3] = dtype(1e-30)
    cells[ny - 1, nx - 1, 7] = dtype(-7 * 2.0 ** -33)
    cells[ny - 2, 0, 8] = dtype(2.0 ** -34)
    return cells, obst


BOXES = [(0, 0, 0, 0), (0, 0, 3, 2), (1, 1, 6, 5), (2, 0, 7, 5), (0, 4, 7, 5), (6, 0, 7, 5), (3, 3, 3, 5)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_restatement_equals_the_formula_in_fractions(dtype, seed):
    nx, ny = 7, 5
    cells, obst = small_case(nx, ny, seed, dtype)
    tilde = F.accelerated(cells, obst, 0.1, 0.005)
    boxes = BOXES + [(0, 0, nx, ny)]
    got = F.force(tilde, obst, boxes)
    want = formula(tilde, obst, boxes)
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (got, want)
    assert np.array_equal(F.force(tilde, obst), want[-1:])


def test_tie_rounds_half_to_even():
    q, bad = F._fixed(np.array([3 * 2.0 ** -33, 5 * 2.0 ** -33, -3 * 2.0 ** -33, 2.0 ** -34, -(2.0 ** -33)]))
    assert list(q) == [2, 2, -2, 0, 0] and not bad.any()


def test_slab_shares_add_up():
    cells, obst = small_case(9, 8, 4, np.float32)
    tilde = F.accelerated(cells, obst, 0.1, 0.005)
    whole = F.force_sums(tilde, obst)[0]
    parts = [F.force_sums(tilde, obst, rows=r)[0] for r in ((0, 3), (3, 4), (4, 8))]
    assert (sum(p[0] for p in parts), sum(p[1] for p in parts)) == whole


def test_nan_stays_in_its_boxes():
    cells, obst = small_case(7, 5, 5, np.float32)
    obst[:] = 0
    obst[1, 1] = 1
    obst[3, 5] = 1
    cells[1, 1, 1] = np.nan                              # leaves solid cell (1, 1) towards (2, 1)
    cells[3, 5, 2] = np.float32(2.0 ** 31)
    tilde = F.accelerated(cells, obst, 0.1, 0.005)
    got = F.force(tilde, obst, [(0, 0, 3, 3), (4, 2, 7, 5), (0, 0, 7, 5), (3, 0, 4, 5)])
    assert np.isnan(got[:3]).all()
    assert np.array_equal(got[3], [0.0, 0.0])
    assert np.array_equal(got, formula(tilde, obst, [(0, 0, 3, 3), (4, 2, 7, 5), (0, 0, 7, 5), (3, 0, 4, 5)]),
                          equal_nan=True)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_momentum_balance_on_the_oracle_step(dtype):
    """P_fluid(t+1) = P~_fluid(t) - F_all(t), up to the collision's rounding and the read-out's
    fixed point: each fluid cell's collision rounds its 9 outputs, each by at most half an ulp of the
    result, so its momentum moves by at most 3 ulp(max f) per component; and each of the at most 16
    values per solid cell is rounded to a multiple of 2^-32, by at most 2^-33."""
    nx, ny, density, accel, omega = 64, 48, 0.1, 0.005, 1.85
    cells, obst = O.random_lattice(nx, ny, 11, dtype=dtype)
    state = cells
    for _ in range(3):
        tilde = F.accelerated(state, obst, density, accel)
        f_all = F.force(tilde, obst)[0]
        p_tilde = np.array(F.fluid_momentum(tilde, obst))
        state, _, _ = O.run(state, obst, 1, density, accel, omega)
        p_new = np.array(F.fluid_momentum(state, obst))
        eps = np.finfo(dtype).eps
        bound = 3 * eps * float(np.abs(state).max()) * int((obst == 0).sum()) + 16 * 2.0 ** -33 * int(obst.sum())
        err = np.abs(p_new - (p_tilde - f_all))
        assert (err <= bound).all(), (err, bound)
        assert err.max() < 1e-3 * np.abs(f_all).max()       # the force is far above the rounding
