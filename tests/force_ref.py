"""Exact CPU restatement of lbm_gpu_obstacle_force (include/lbm_gpu.h) in Python ints: the
momentum-exchange force on the solid cells of each box, from the lattice f~ that the next step
streams.  TEST INFRASTRUCTURE ONLY."""
import ctypes as C

import numpy as np

import oracle_lib as O

FIX = 32                                   # each value enters as round_half_even(v * 2^32)
LIMIT = 2.0 ** 31                          # ... or marks its box NaN when not finite or this large
# speed vectors in the header's order (+y = towards row ny-1) and the opposite speeds
CK = [(0, 0), (1, 0), (0, 1), (-1, 0), (0, -1), (1, 1), (-1, 1), (-1, -1), (1, -1)]
OPP = [0, 3, 4, 1, 2, 7, 8, 5, 6]


def accelerated(cells, obst, density, accel):
    """f~: the lattice with row ny-2 accelerated by the oracle's accelerate_flow (fp32 or fp64;
    for a binary16 lattice pass the decoded fp32 values)."""
    a = np.ascontiguousarray(cells).copy()
    ny, nx, _ = a.shape
    ct, sfx = (C.c_double, "f64") if a.dtype == np.float64 else (C.c_float, "f32")
    fn = getattr(O.oracle(), "oracle_accelerate_flow_" + sfx)
    fn.argtypes = [C.c_int, C.c_int, ct, ct, C.c_void_p, C.c_void_p]
    fn.restype = None
    o = np.ascontiguousarray(obst, dtype=np.int32)
    fn(nx, ny, density, accel, a.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p))
    return a


def _at(a, dx, dy):
    """a at (x + dx, y + dy), periodic in both directions."""
    return np.roll(a, shift=(-dy, -dx), axis=(0, 1))


def _fixed(v):
    """(round_half_even(v * 2^32) as int64, mark) per value; marked values give 0."""
    v = np.asarray(v, dtype=np.float64)
    ok = np.abs(v) < LIMIT                 # False for NaN too
    q = np.rint(np.ldexp(np.where(ok, v, 0.0), FIX)).astype(np.int64)
    return q, ~ok


def _exact_sum(q):
    """Sum of an int64 array as a Python int (halves summed apart, so nothing wraps)."""
    q = np.asarray(q, dtype=np.int64)
    return int(np.sum(q >> 32, dtype=np.int64)) * (1 << 32) + int(np.sum(q & 0xFFFFFFFF, dtype=np.int64))


def force_sums(tilde, obst, boxes=None, rows=None):
    """Exact integer sums [(Sx, Sy) or None if marked] per box, in units of 2^-32.  tilde: (ny, nx, 9)
    f~; obst: (ny, nx); boxes: (n, 4) {x0, y0, x1, y1} or None for the whole grid; rows: (r0, r1) to
    count only the solid cells of those rows (a slab handle's share)."""
    tilde = np.asarray(tilde)
    ny, nx, _ = tilde.shape
    solid = np.asarray(obst) != 0
    boxes = [(0, 0, nx, ny)] if boxes is None else [tuple(int(v) for v in b) for b in np.asarray(boxes).reshape(-1, 4)]
    ys, xs = np.mgrid[0:ny, 0:nx]
    keep = np.ones((ny, nx), dtype=bool)
    if rows is not None:
        keep = (ys >= rows[0]) & (ys < rows[1])
    out = []
    links = []
    for d in range(1, 9):
        dx, dy = CK[d]
        link = solid & ~_at(solid, dx, dy) & keep
        qa, ba = _fixed(tilde[:, :, d])                          # f~_d(x_s): leaves the solid
        qb, bb = _fixed(_at(tilde[:, :, OPP[d]], dx, dy))        # f~_opp(d)(x_s + c_d): streams in
        links.append((dx, dy, link, qa, ba, qb, bb))
    for (x0, y0, x1, y1) in boxes:
        inbox = (xs >= x0) & (xs < x1) & (ys >= y0) & (ys < y1)
        sx = sy = 0
        bad = False
        for dx, dy, link, qa, ba, qb, bb in links:
            sel = link & inbox
            if not sel.any():
                continue
            bad = bad or bool(ba[sel].any() or bb[sel].any())
            q = _exact_sum(qa[sel]) + _exact_sum(qb[sel])
            sx -= dx * q
            sy -= dy * q
        out.append(None if bad else (sx, sy))
    return out


def to_double(s):
    """The correctly rounded double of S * 2^-32 (Python's int / int rounds once)."""
    return s / (1 << FIX)


def force(tilde, obst, boxes=None, rows=None):
    """(n, 2) float64: lbm_gpu_obstacle_force's output for f~."""
    sums = force_sums(tilde, obst, boxes, rows)
    return np.array([[np.nan, np.nan] if s is None else [to_double(s[0]), to_double(s[1])] for s in sums],
                    dtype=np.float64)


def fluid_momentum(cells, obst):
    """(P_x, P_y) of the fluid cells, summed in float64."""
    f = np.asarray(cells, dtype=np.float64)[np.asarray(obst) == 0]
    cx = np.array([c[0] for c in CK], dtype=np.float64)
    cy = np.array([c[1] for c in CK], dtype=np.float64)
    return float(np.sum(f @ cx)), float(np.sum(f @ cy))
