"""Exact CPU restatements of the device read-outs' integer arithmetic, in Python ints:
the fixed-point |u| sum behind av_velocity and av_vels, the host's conversion of that sum
to an average, and the fixed-point mass of the digest.  TEST INFRASTRUCTURE ONLY."""
import platform

import numpy as np

import lbm_b200 as L
import oracle_f16 as H
import oracle_lib as O

FIX_BITS = 52            # LBM_FIX_SCALE = 2^52 (csrc/lbm_kernels.cuh)
SPEED_LIMIT = 2.0        # LBM_SPEED_LIMIT: a fluid |u| not below it (or NaN) makes the average NaN
MASS_BITS = 32           # lbm_digest: mass = sum of round(f * 2^32)
MASS_LIMIT = 2.0 ** 31   # a value of this magnitude (or non-finite) has no fixed-point mass


def _halves_sum(q):
    """Exact sum of a uint64 array as a Python int: the high and low 32-bit halves are summed
    separately, so that no partial sum can wrap."""
    q = np.ascontiguousarray(q, dtype=np.uint64).ravel()
    lo = int(np.sum(q & np.uint64(0xFFFFFFFF), dtype=np.uint64))
    hi = int(np.sum(q >> np.uint64(32), dtype=np.uint64))
    return (hi << 32) + lo


def fixed_u_sum(u, obst):
    """S = sum over fluid cells of rint(float64(u) * 2^52) (to_fixed, round half to even), for
    fp32 or fp64 u; obstacle cells add nothing.  None when a fluid |u| is NaN or not below
    LBM_SPEED_LIMIT: the device marks the sum instead and reports NaN."""
    u = np.asarray(u)
    fluid = np.asarray(obst) == 0
    v = u[fluid].astype(np.float64)
    if not np.all(v < SPEED_LIMIT):
        return None
    return _halves_sum(np.rint(np.ldexp(v, FIX_BITS)).astype(np.uint64))


def _round_significand(n, bits):
    """The non-negative int n rounded to `bits` significant bits, ties to even."""
    extra = n.bit_length() - bits
    if extra <= 0:
        return n
    q, r = divmod(n, 1 << extra)
    half = 1 << (extra - 1)
    if r > half or (r == half and q & 1):
        q += 1
    return q << extra


def long_double_bits():
    """Significand bits of the host's long double: x87 extended on x86-64, binary128 on
    aarch64."""
    return 113 if platform.machine() in ("aarch64", "arm64") else 64


def host_average(S, n, dtype):
    """The host's average of a fixed-point sum S over n cells (run_impl, lbm_gpu_av_velocity):
    (long double)S / 2^52, converted to double, divided by n in double, then cast to dtype.
    S = None (a marked sum) gives NaN."""
    if S is None:
        return dtype(np.nan)
    s = float(_round_significand(int(S), long_double_bits()))      # long double, then double
    with np.errstate(invalid="ignore", divide="ignore"):          # n = 0: 0/0, as in C
        return dtype(np.float64(np.ldexp(s, -FIX_BITS)) / np.float64(n))


def digest_mass(cells):
    """total_density of lbm_gpu_digest: sum of rint(float64(f) * 2^32) over every cell and speed,
    wrapped mod 2^64, read as int64 and divided by 2^32.  NaN when a value is non-finite or of
    magnitude 2^31 or more."""
    flat = np.asarray(cells).ravel()
    m = 0
    for i in range(0, flat.size, 1 << 22):         # a few million values at a time (large grids)
        f = flat[i:i + (1 << 22)].astype(np.float64)
        if not np.all(np.abs(f) < MASS_LIMIT):
            return float("nan")
        m += _halves_sum(np.rint(np.ldexp(f, MASS_BITS)).astype(np.int64).view(np.uint64))
    m &= (1 << 64) - 1
    if m >= 1 << 63:
        m -= 1 << 64
    return float(m) / 2.0 ** MASS_BITS


def checksum(cells, chunk_rows=256):
    """L.lattice_checksum of the whole lattice, taken a few rows at a time (large grids)."""
    total = 0
    for r in range(0, cells.shape[0], chunk_rows):
        total += L.lattice_checksum(cells[r:r + chunk_rows], global_row0=r)
    return total & ((1 << 64) - 1)


def digest(cells):
    """(total_density, checksum) as lbm_gpu_digest gives them for this lattice."""
    return digest_mass(cells), checksum(cells)


def strict_step_speeds(cells, obst, density, accel, omega):
    """One strict timestep of the oracle: (the new lattice, the per-cell |u| that the strict
    kernels add to av_vels).  The strict cell_update computes |u| from the values it stores with
    cell_macroscopic's expression tree, and an obstacle cell gives 0: that is final_state's |u|
    of the new lattice.  For STORE_F16 pass the decoded lattice; the new lattice is returned
    before it is encoded, which is where the f16 kernels take |u| from."""
    obst = np.ascontiguousarray(obst, dtype=np.int32)
    new, _, _ = O.run(cells, obst, 1, density, accel, omega)
    return new, O.final_state(new, obst, density)[2]


def strict_av_vels(cells, obst, steps, density, accel, omega, f16=False):
    """(final lattice, av_vels) of a strict run, av_vels bit for bit as the device reports them.
    With f16 the lattice is kept encoded between steps, as oracle_f16.run_f16 does."""
    dtype = np.float64 if cells.dtype == np.float64 else np.float32
    n = int((np.asarray(obst) == 0).sum())
    av = np.empty(steps, dtype=dtype)
    state = H.f16_encode(cells, density) if f16 else cells
    for t in range(steps):
        src = H.f16_decode(state, density) if f16 else state
        new, speeds = strict_step_speeds(src, obst, density, accel, omega)
        av[t] = host_average(fixed_u_sum(speeds, obst), n, dtype)
        state = H.f16_encode(new, density) if f16 else new
    return (H.f16_decode(state, density) if f16 else state), av
