"""CPU only: the restatement of lbm_gpu_coarse_fields' arithmetic (tests/coarse_ref.py) against
a slow, obviously exact one in Python ints and fractions.Fraction."""
import math
from fractions import Fraction

import numpy as np
import pytest

import coarse_ref as CR


def slow_coarse(v, factor):
    """Block means of v by the definition: every cell's exact round-half-even of v * 2^32, an
    exact integer sum, one rounding of the double division, one rounding to float32."""
    ny, nx = v.shape
    out = np.empty((-(-ny // factor), -(-nx // factor)), dtype=np.float32)
    for J in range(out.shape[0]):
        for C in range(out.shape[1]):
            blk = v[J * factor:(J + 1) * factor, C * factor:(C + 1) * factor]
            s, bad = 0, False
            for x in blk.ravel():
                x = float(x)
                if not (abs(x) < 2.0 ** 15):
                    bad = True
                    continue
                s += round(Fraction(x) * 2 ** 32)            # round() of a Fraction: half to even
            if bad:
                out[J, C] = np.nan
                continue
            d = float(s) * 2.0 ** -32 / float(blk.size)      # float(int): nearest, ties to even
            out[J, C] = np.float32(d)
    return out


def same(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    u = {2: np.uint16, 4: np.uint32}[a.dtype.itemsize]
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(u), b[~nb].view(u))


@pytest.mark.parametrize("factor", [2, 3, 4, 7, 16])
@pytest.mark.parametrize("shape", [(23, 37), (1, 9), (5, 1), (16, 16)])
def test_block_means_match_the_definition(factor, shape):
    rng = np.random.default_rng(factor * 100 + shape[0])
    v = (rng.standard_normal(shape) * 10.0 ** rng.integers(-12, 3, size=shape)).astype(np.float32)
    got = CR.mean(*CR.block_sums(v, factor), CR.block_cells(*shape, factor))
    assert same(got, slow_coarse(v, factor))


def test_ties_round_to_even_and_tiny_values_vanish():
    v = np.array([[2.0 ** -33, 3 * 2.0 ** -33, -2.0 ** -33, 1e-30]], dtype=np.float32)
    S, B = CR.block_sums(v, 4)
    assert S[0, 0] == 0 + 2 + 0 + 0 and not B[0, 0]


def test_the_bound_and_non_finite_values_mark_only_their_block():
    v = np.zeros((4, 6), dtype=np.float32)
    v[0, 0] = 2.0 ** 15
    v[3, 5] = np.nan
    v[2, 2] = np.float32(2.0 ** 15 - 2.0 ** -8)              # the largest value below the bound
    m = CR.mean(*CR.block_sums(v, 2), CR.block_cells(4, 6, 2))
    assert np.isnan(m[0, 0]) and np.isnan(m[1, 2])
    assert np.isfinite(np.delete(m.ravel(), [0, 5])).all()
    assert m[1, 1] == np.float32((2.0 ** 15 - 2.0 ** -8) / 4)


def test_largest_block_sum_stays_in_int64():
    v = np.full((256, 256), np.float32(-(2.0 ** 15 - 2.0 ** -8)), dtype=np.float32)
    S, B = CR.block_sums(v, 256)
    assert int(S[0, 0]) == -(2 ** 47 - 2 ** 24) * 2 ** 16 and not B[0, 0]
    assert math.isclose(float(CR.mean(S, B, CR.block_cells(256, 256, 256))[0, 0]), -(2.0 ** 15 - 2.0 ** -8))


def test_binary16_pressure_is_shifted():
    d = 0.1
    p = np.array([[CR.p0(d), CR.p0(d) + np.float32(1e-5)]], dtype=np.float32)
    h = CR.to_f16((p, p, p, p), d)[3]
    assert h[0, 0] == 0 and h[0, 1] == np.float16(np.float32(p[0, 1] - CR.p0(d)))
    assert abs(CR.decode_pressure(h, d)[0, 1] - p[0, 1]) < 3e-8          # 11 bits of 1e-5, and the fp32 add
