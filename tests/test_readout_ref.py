"""The read-out restatements of tests/readout_ref.py against exact rational arithmetic
(fractions.Fraction) on random inputs: sums beyond 2^64, ties of the rounding to integers,
speeds below 2^-29 where rounding decides, and the host's long double conversion.  CPU only."""
from fractions import Fraction

import numpy as np
import pytest

import readout_ref as R


def _rint(x):
    """Round half to even of an exact rational (round() of a Fraction)."""
    return round(x)


def _to_double(x):
    """An exact non-negative rational to the nearest double, ties to even."""
    if x == 0:
        return 0.0
    e = x.numerator.bit_length() - x.denominator.bit_length()
    while Fraction(2) ** e > x:
        e -= 1
    while Fraction(2) ** (e + 1) <= x:
        e += 1
    ulp = Fraction(2) ** (e - 52)
    return float(_rint(x / ulp) * ulp)


def exact_fixed_u_sum(u, obst):
    return sum(_rint(Fraction(float(v)) * 2 ** 52) for v, o in zip(np.ravel(u), np.ravel(obst)) if o == 0)


def exact_host_average(S, n, dtype):
    bits = R.long_double_bits()
    e = max(S.bit_length() - bits, 0)
    ld = _rint(Fraction(S, 2 ** e)) * 2 ** e                    # (long double)S
    d = _to_double(Fraction(ld, 2 ** 52))                        # (double)(S / 2^52)
    return dtype(_to_double(Fraction(d) / n))                     # / n in double, then the cast


def _speeds(rng, n, dtype):
    u = np.concatenate([
        rng.uniform(0, 1.99, n),                                  # ordinary speeds
        rng.uniform(0, 2.0 ** -29, n // 4),                       # where the rounding to 2^-52 decides
        np.ldexp(rng.integers(0, 64, n // 8) + 0.5, -52),          # exact ties: k + 1/2 units
        [0.0, np.nextafter(dtype(2), dtype(0)), 2.0 ** -53, 3 * 2.0 ** -53, 5 * 2.0 ** -54],
    ]).astype(dtype)
    obst = (rng.random(u.size) < 0.2).astype(np.int32)
    return u, obst


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("seed", range(4))
def test_fixed_u_sum_is_exact(dtype, seed):
    rng = np.random.default_rng(seed)
    u, obst = _speeds(rng, 3000, dtype)
    assert R.fixed_u_sum(u, obst) == exact_fixed_u_sum(u, obst)


def test_fixed_u_sum_beyond_64_bits():
    """2^13 cells just below the speed limit: the sum is above 2^65, each term near 2^53."""
    u = np.full(1 << 13, np.nextafter(2.0, 0), dtype=np.float64)
    obst = np.zeros(u.size, dtype=np.int32)
    S = R.fixed_u_sum(u, obst)
    assert S > 2 ** 64 and S == exact_fixed_u_sum(u, obst)
    assert S == u.size * (2 ** 53 - 1)


def test_fixed_u_sum_rounds_half_to_even():
    u = np.ldexp(np.array([0.5, 1.5, 2.5, 3.5, 0.25, 0.75]), -52)
    assert R.fixed_u_sum(u, np.zeros(u.size, np.int32)) == 0 + 2 + 2 + 4 + 0 + 1


def test_fixed_u_sum_refuses_what_the_device_marks():
    obst = np.zeros(3, np.int32)
    for bad in (np.nan, 2.0, np.inf, 1e30):
        assert R.fixed_u_sum(np.array([0.1, bad, 0.2], np.float32), obst) is None
    # an obstacle cell is never looked at
    assert R.fixed_u_sum(np.array([0.1, np.nan, 0.2], np.float32), np.array([0, 1, 0], np.int32)) is not None


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("seed", range(6))
def test_host_average_is_the_long_double_conversion(dtype, seed):
    rng = np.random.default_rng(100 + seed)
    b = R.long_double_bits()
    for _ in range(200):
        bits = int(rng.integers(30, 128))
        S = int.from_bytes(rng.bytes(16), "little") >> (128 - bits)
        if rng.random() < 0.3:          # an exact tie at the long double's last place
            k = int(rng.integers(1, 10))
            m = (int.from_bytes(rng.bytes(16), "little") >> (128 - b)) | (1 << (b - 1))
            S = (m << k) | (1 << (k - 1))
        n = int(rng.integers(1, 1 << 34))
        want = exact_host_average(S, n, dtype)
        got = R.host_average(S, n, dtype)
        assert np.array_equal(np.array(got, dtype), np.array(want, dtype)), (S, n)


def test_host_average_ties_of_the_long_double():
    """S with more significant bits than the long double has, at an exact tie: rounds to even."""
    b = R.long_double_bits()
    for odd in (0, 1):
        S = ((1 << (b - 1)) + odd) << 8 | (1 << 7)
        assert R._round_significand(S, b) == (((1 << (b - 1)) + odd + odd) << 8)
        assert R.host_average(S, 3, np.float64) == exact_host_average(S, 3, np.float64)


def test_host_average_of_a_marked_sum_or_no_cells_is_nan():
    assert np.isnan(R.host_average(None, 10, np.float32))
    assert np.isnan(R.host_average(0, 0, np.float64))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_digest_mass_is_exact_and_wraps_like_int64(dtype):
    rng = np.random.default_rng(7)
    cells = rng.uniform(-0.5, 1.5, size=(13, 17, 9)).astype(dtype)
    cells[0, 0, :3] = np.ldexp(np.array([0.5, 1.5, -2.5]), -32)    # ties of the rounding
    exact = sum(_rint(Fraction(float(f)) * 2 ** 32) for f in cells.ravel())
    assert R.digest_mass(cells) == float(exact) / 2 ** 32
    # terms near 2^63: the 64-bit sum wraps and is read as int64, as on the device
    big = np.full((4, 1, 9), np.nextafter(2.0 ** 31, 0), dtype=np.float64)
    exact = sum(_rint(Fraction(float(f)) * 2 ** 32) for f in big.ravel()) % 2 ** 64
    exact = exact - 2 ** 64 if exact >= 2 ** 63 else exact
    assert R.digest_mass(big) == float(exact) / 2 ** 32


def test_digest_mass_of_what_has_no_fixed_point_value_is_nan():
    for bad in (np.nan, np.inf, -np.inf, 2.0 ** 31, -3e9):
        cells = np.full((2, 2, 9), 0.1, np.float32)
        cells[1, 0, 4] = bad
        assert np.isnan(R.digest_mass(cells))


def test_chunked_checksum_is_the_whole_checksum():
    rng = np.random.default_rng(3)
    cells = rng.uniform(0, 1, size=(37, 11, 9)).astype(np.float32)
    import lbm_b200 as L
    assert R.checksum(cells, chunk_rows=5) == L.lattice_checksum(cells)
