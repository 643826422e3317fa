"""Reference and error bound of ONE timestep of the default build.  TEST INFRASTRUCTURE ONLY.

f64_step   the step computed in extended precision (np.longdouble: 64 significand bits on
           x86-64, 113 on aarch64) from the GPU's own previous state.  The accelerated source
           comes from oracle_lib.timestep in the lattice's own precision: both builds apply
           accelerate_flow with the same single rounded add/sub, so it is exact, not an error
           source.  Propagation and the BGK collision are then evaluated as plain formulas.
bound      a per-speed bound on |default step - exact step|, derived below, and a bound on
           each fluid cell's |u| as the default build adds it to av_vels.
collide_fast_emulated
           a numpy float32 restatement of collide_fast (csrc/lbm_kernels.cuh), operation for
           operation, with the approximate hardware instructions moved by their largest
           documented error; test_default_ref.py checks that bound() holds for it and that
           small mistakes in the collision exceed it.

Derivation (eps = 2^-24 for fp32, 2^-53 for fp64; first order in eps; P = sum_k |p_k| of
the pulled values, rho = sum_k p_k, j = rho u; v = the velocity component of direction k,
v = c_k . u).  collide_fast computes, with every operation rounded once:

  e, w, n, s   two adds each; rho = ((p0+p2)+(p4+e))+w: no leaf goes through more than 5
               roundings, so |d rho| <= 5 eps P.
  ninv         -1/rho: rcp.approx (1 ulp, relative 2 eps) plus one Newton step
               fma(nr, fma(x, nr, 1), nr), which leaves a relative error of eps (1 + 6 eps).
  ux = (w-e)*ninv
               the computed ux times the computed rho is j_x (1 + 2 theta) + d(w-e), so
               |d j_x| <= eps (2 P_x + 3 |j_x|) with P_x the |p| of the six speeds with an x
               component (<= P); the same for y.  Hence |d j_k| <= eps (2 P + 3 |rho| |v|) on
               the axes, eps (4 P + 4.25 |rho| |u|) on the diagonals (3 sqrt 2 < 4.25), and
               the vector |d j| <= eps (4 P + 4.25 |rho| |u|).
  c_k          = (1-w) p_k + f_k(rho, j),  f_k = om w_k (rho + 3 j_k + 4.5 j_k^2/rho - 1.5 |j|^2/rho).
               Propagated input error:
                 |df_k| <= om w_k [ (1 + 4.5 v^2 + 1.5 u^2) |d rho| + (3 + 9|v|) |d j_k| + 3 |u| |d j| ].
               Evaluation error, counting the roundings each term passes through (the
               products with rho*ow_k, 3, 4.5, the two inner fmas, the final fma, and the two
               roundings of the constant ow_k = fl(omega * fl(w_k))):
                 4.5 v^2: 7,  3 |v|: 7,  base = 1 - 1.5 u^2: 7 |base| + the 3 u^2 of fl(u^2),
                 the diagonals' fl(ux +- uy): 3 |v| + 9 v^2 more,
                 the final fma: eps |1-omega| |p_k| (1 - omega is exact for 0.5 <= omega <= 2;
                 outside that range its rounding adds the same again).
               So, per speed (rest speed k = 0 with v = 0 is covered by the axis line):
                 axis      eps om w_k |rho| (7 + 21|v| + 31.5 v^2 + 13.5 u^2)
                 diagonal  eps om w_k |rho| (7 + 24|v| + 40.5 v^2 + 13.5 u^2)
               plus the propagated terms above and eps |1-omega| |p_k|.
  |u|          av_vels takes |u| from the PULLED values (DESIGN.md section 4): sqrt of
               fma(uy, uy, ux*ux).  | |u computed| - |u| | <= |d ux| + |d uy| +
               (eps + sqrt error) |u|, with |d u_x| <= eps (2 P_x + (3 + 5 P/|rho|) |j_x|)/|rho|;
               sqrt.approx.ftz.f32 has a relative error of at most 2^-23 (PTX ISA), the
               fp64 sqrt is correctly rounded (eps), and a flushed subnormal u^2 can lose
               2^-63.
  obstacles    bounce-back is a permutation of the pulled values: the bound is exactly 0.

Every coefficient is derived, none fitted; HIGHER_ORDER covers the O(eps^2) terms, which are
below 2^-20 of the first-order ones wherever eps P / |rho| < 2^-20 (the test domains stay far
inside that).
"""
import numpy as np

import oracle_lib as O

EPS32 = 2.0 ** -24
EPS64 = 2.0 ** -53
SQRT_APPROX_REL = 2.0 ** -23      # sqrt.approx.f32: largest relative error (PTX ISA)
HIGHER_ORDER = 1.0 + 2.0 ** -10

CX = np.array([0, 1, 0, -1, 0, 1, -1, -1, 1])
CY = np.array([0, 0, 1, 0, -1, 1, 1, -1, -1])
WEIGHTS = np.array([4 / 9] + [1 / 9] * 4 + [1 / 36] * 4)
OPPOSITE = [0, 3, 4, 1, 2, 7, 8, 5, 6]
XDIR = [1, 5, 8, 3, 6, 7]          # speeds with an x component
YDIR = [2, 5, 6, 4, 7, 8]


def eps_of(dtype):
    return EPS64 if np.dtype(dtype) == np.float64 else EPS32


def pull(src):
    """p[y, x, k] = src[y - cy_k, x - cx_k, k], periodic: the values cell (x, y) collides."""
    p = np.empty_like(src)
    for k in range(9):
        p[:, :, k] = np.roll(src[:, :, k], (CY[k], CX[k]), axis=(0, 1))
    return p


def macroscopic(p):
    """(rho, ux, uy, P) of pulled values p[..., 9] in p's own precision."""
    rho = p.sum(axis=-1)
    jx = p[..., 1] + p[..., 5] + p[..., 8] - (p[..., 3] + p[..., 6] + p[..., 7])
    jy = p[..., 2] + p[..., 5] + p[..., 6] - (p[..., 4] + p[..., 7] + p[..., 8])
    with np.errstate(divide="ignore", invalid="ignore"):
        return rho, jx / rho, jy / rho, np.abs(p).sum(axis=-1)


def collide_exact(p, omega):
    """BGK collision of pulled values p[..., 9] evaluated in p's precision as the plain formula
    c_k = (1 - omega) p_k + omega w_k rho (1 + 3 u_k + 4.5 u_k^2 - 1.5 u^2)."""
    rho, ux, uy, _ = macroscopic(p)
    one = p.dtype.type(1)
    usq = ux * ux + uy * uy
    c = np.empty_like(p)
    for k in range(9):
        uk = CX[k] * ux + CY[k] * uy
        w = p.dtype.type(4 if k == 0 else 1) / p.dtype.type(9 if k < 5 else 36)
        c[..., k] = (one - omega) * p[..., k] + omega * w * rho * (
            one + 3 * uk + p.dtype.type(4.5) * uk * uk - p.dtype.type(1.5) * usq)
    return c


def f64_step(cells, obst, density, accel, omega):
    """One default step from `cells` (float32 or float64, the GPU's state) in extended
    precision.  Returns a dict: cells (the new lattice, longdouble), pulled (longdouble),
    rho, ux, uy, speed (|u| of the pulled values; 0 at obstacles), P, obst, omega (the
    lattice-precision omega as longdouble)."""
    dtype = cells.dtype.type
    obst = np.asarray(obst) != 0
    src, _, _ = O.timestep(cells, obst.astype(np.int32), density, accel, omega)
    p = pull(src).astype(np.longdouble)
    om = np.longdouble(dtype(omega))
    new = collide_exact(p, om)
    new[obst] = p[obst][:, OPPOSITE]
    rho, ux, uy, P = macroscopic(p)
    speed = np.sqrt(ux * ux + uy * uy)
    speed[obst] = 0
    return dict(cells=new, pulled=p, rho=rho, ux=ux, uy=uy, speed=speed, P=P, obst=obst, omega=om)


def bound(p, omega, eps, obst=None, sqrt_rel=None):
    """(per-speed bound [..., 9], per-cell |u| bound [...]) on the error of one default
    collision of the pulled values p (see the module docstring).  omega as the lattice holds
    it; eps 2^-24 (fp32) or 2^-53 (fp64); sqrt_rel defaults to sqrt.approx's error for fp32 and
    to eps for fp64.  Obstacle cells get 0."""
    p = np.asarray(p, dtype=np.float64)
    om = float(omega)
    if sqrt_rel is None:
        sqrt_rel = SQRT_APPROX_REL if eps > EPS64 else eps
    rho, ux, uy, P = macroscopic(p)
    ar = np.abs(rho)
    usq = ux * ux + uy * uy
    u = np.sqrt(usq)
    keep = abs(1.0 - om) * (1.0 if 0.5 <= om <= 2.0 else 2.0)
    dj_vec = 4 * P + 4.25 * ar * u
    out = np.empty(p.shape, dtype=np.float64)
    for k in range(9):
        v = CX[k] * ux + CY[k] * uy
        av = np.abs(v)
        diag = k >= 5
        ev = 7 + (24 if diag else 21) * av + (40.5 if diag else 31.5) * v * v + 13.5 * usq
        dj_k = dj_vec if diag else 2 * P + 3 * ar * av
        prop = 5 * P * (1 + 4.5 * v * v + 1.5 * usq) + (3 + 9 * av) * dj_k + 3 * u * dj_vec
        out[..., k] = keep * np.abs(p[..., k]) + om * WEIGHTS[k] * (ar * ev + prop)
    out *= HIGHER_ORDER * eps
    px = np.abs(p[..., XDIR]).sum(axis=-1)
    py = np.abs(p[..., YDIR]).sum(axis=-1)
    with np.errstate(divide="ignore", invalid="ignore"):
        spd = eps * (2 * (px + py) + (3 + 5 * P / ar) * ar * (np.abs(ux) + np.abs(uy))) / ar
    spd = HIGHER_ORDER * (spd + (eps + sqrt_rel) * u) + 2.0 ** -63
    if obst is not None:
        o = np.asarray(obst) != 0
        out[o] = 0
        spd[o] = 0
    return out, spd


def av_bound(speed, speed_bound, obst, eps):
    """Bound on |av_vels - exact mean |u||: the cells' bounds, the float sums of the four cells
    of a quad (two roundings of at most eps each, relative to the quad's sum), the 2^-52
    fixed point, and the host's division and cast (eps of the result)."""
    fluid = np.asarray(obst) == 0
    n = max(int(fluid.sum()), 1)
    s = np.asarray(speed, dtype=np.float64)[fluid]
    mean = s.sum() / n
    return (np.asarray(speed_bound)[fluid].sum() + 2 * eps * s.sum()) / n + 2 * eps * mean + 2.0 ** -52


# ------------------------------------------------------------------ float32 restatement
def _fma(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _rcp_approx(x, sign):
    """rcp.approx.ftz.f32: the correctly rounded reciprocal moved by sign (-1, 0, +1) ulps, the
    largest error the PTX ISA documents (1 ulp)."""
    r = (1.0 / x.astype(np.float64)).astype(np.float32)
    return np.where(sign > 0, np.nextafter(r, np.float32(np.inf)),
                    np.where(sign < 0, np.nextafter(r, np.float32(-np.inf)), r)).astype(np.float32)


def _sqrt_approx(x, sign):
    """sqrt.approx.ftz.f32: a float32 within SQRT_APPROX_REL of the true root, as far from it
    as that allows in direction sign."""
    t = np.sqrt(np.maximum(x.astype(np.float64), 0.0))
    r = (t * (1.0 + sign * SQRT_APPROX_REL)).astype(np.float32)
    off = np.abs(r.astype(np.float64) - t) > SQRT_APPROX_REL * t
    r = np.where(off, np.nextafter(r, t.astype(np.float32)), r)
    return np.where(x < 0, np.float32(np.nan), r).astype(np.float32)


def collide_fast_emulated(p, omega, rng=None, perturb=None):
    """collide_fast (csrc/lbm_kernels.cuh) on float32 pulled values p[..., 9]: returns (c, |u|).
    The approximate instructions take their largest documented error in a random direction
    per cell (rng) or none (rng None).  `perturb` names a deliberate mistake, for checking that
    bound() would notice it: 'ow0', 'ow1', 'ow2', 'f45', 'm15' (that constant off by 2^-18
    relative), 'swap' (ux and uy exchanged in direction 2), 'usq' (u^2 without uy^2)."""
    f = np.float32
    p = np.asarray(p, dtype=f)
    om = f(omega)
    rel = f(1 + 2.0 ** -18)
    keep = f(1) - om
    ow0 = om * f(4.0 / 9.0) * (rel if perturb == "ow0" else f(1))
    ow1 = om * f(1.0 / 9.0) * (rel if perturb == "ow1" else f(1))
    ow2 = om * f(1.0 / 36.0) * (rel if perturb == "ow2" else f(1))
    f45 = f(4.5) * (rel if perturb == "f45" else f(1))
    m15 = f(-1.5) * (rel if perturb == "m15" else f(1))
    shape = p.shape[:-1]
    if rng is None:
        s_rcp = s_sqrt = np.zeros(shape)
    else:
        s_rcp = rng.integers(-1, 2, size=shape)
        s_sqrt = rng.choice([-1.0, 1.0], size=shape)
    q = [p[..., k] for k in range(9)]
    e = (q[1] + q[5]) + q[8]
    w = (q[3] + q[6]) + q[7]
    n = (q[2] + q[5]) + q[6]
    s = (q[4] + q[7]) + q[8]
    rho = ((q[0] + q[2]) + (q[4] + e)) + w
    with np.errstate(all="ignore"):
        nr = _rcp_approx(-rho, s_rcp)
        ninv = _fma(nr, _fma(rho, nr, np.full(shape, f(1))), nr)
        ux = (w - e) * ninv
        uy = (s - n) * ninv
        usq = ux * ux if perturb == "usq" else _fma(uy, uy, ux * ux)
        base = _fma(np.full(shape, m15), usq, np.full(shape, f(1)))
        r1, r2 = rho * ow1, rho * ow2
        b0 = (rho * ow0) * base
        b1, l1, n1, q1 = r1 * base, r1 * f(3), r1 * f(-3), r1 * f45
        b2, l2, n2, q2 = r2 * base, r2 * f(3), r2 * f(-3), r2 * f45
        upv, umv = ux + uy, ux - uy
        c = np.empty(p.shape, dtype=f)
        kp = np.full(shape, keep)
        c[..., 0] = _fma(kp, q[0], b0)

        def d(k, u, lin, quad, b):
            c[..., k] = _fma(kp, q[k], _fma(u, _fma(np.broadcast_to(quad, shape), u, lin), b))
        d(1, ux, l1, q1, b1)
        d(3, ux, n1, q1, b1)
        d(2, ux if perturb == "swap" else uy, l1, q1, b1)
        d(4, uy, n1, q1, b1)
        d(5, upv, l2, q2, b2)
        d(7, upv, n2, q2, b2)
        d(8, umv, l2, q2, b2)
        d(6, umv, n2, q2, b2)
        speed = _sqrt_approx(usq, s_sqrt)
    return c, speed
