"""The default build's per-step error bound (default_ref.py) is sound and tight on the CPU:
the float32 restatement of collide_fast stays within it on about 10^6 cells drawn from the
domains the GPU tests use, and each of a set of small mistakes in the collision exceeds it.
Without the second half, the GPU test that holds every step to the bound could pass with a
bound too loose to catch anything."""
import numpy as np
import pytest

import default_ref as R
import oracle_lib as O

OMEGAS = [0.5, 1.0, 1.5, 1.85, 1.99]
DENSITIES = [0.01, 0.1, 1.0]


def sample_cells(n, seed):
    """n pulled cells per (omega, density) pair: equilibria with |u| up to about 1.5 (which have
    negative speeds from |u| ~ 0.6 on), scaled by random factors, and on a third of the cells
    random negative and positive offsets of up to 30 % of the density."""
    rng = np.random.default_rng(seed)
    out = []
    for omega in OMEGAS:
        for density in DENSITIES:
            rho = density * rng.uniform(0.5, 1.5, n)
            speed = 1.5 * rng.random(n) ** 2
            ang = rng.uniform(0, 2 * np.pi, n)
            ux, uy = speed * np.cos(ang), speed * np.sin(ang)
            p = np.empty((n, 9))
            for k in range(9):
                uk = R.CX[k] * ux + R.CY[k] * uy
                p[:, k] = R.WEIGHTS[k] * rho * (1 + 3 * uk + 4.5 * uk * uk - 1.5 * (ux * ux + uy * uy))
            p *= rng.uniform(0.7, 1.3, (n, 9))
            noisy = rng.random(n) < 1 / 3
            p[noisy] += density * rng.uniform(-0.3, 0.3, (int(noisy.sum()), 9))
            p = p.astype(np.float32)
            r, vx, vy, _ = R.macroscopic(p.astype(np.float64))
            keep = (np.abs(r) > 0.2 * density) & (np.hypot(vx, vy) < 1.6)
            out.append((omega, p[keep]))
    return out


@pytest.fixture(scope="module")
def samples():
    return sample_cells(70_000, seed=1)


def ratios(samples, perturb=None):
    """Largest |emulated - exact| / bound over the sample, for the lattice and for |u|."""
    rng = np.random.default_rng(2)
    worst_c = worst_u = 0.0
    for omega, p in samples:
        om32 = np.float32(omega)
        c, u = R.collide_fast_emulated(p, om32, rng=rng, perturb=perturb)
        pe = p.astype(np.longdouble)
        exact = R.collide_exact(pe, np.longdouble(om32))
        rho, ux, uy, _ = R.macroscopic(pe)
        b, bu = R.bound(p, om32, R.EPS32)
        err = np.abs(c.astype(np.longdouble) - exact).astype(np.float64)
        err_u = np.abs(u.astype(np.longdouble) - np.sqrt(ux * ux + uy * uy)).astype(np.float64)
        worst_c = max(worst_c, float(np.max(err / b)))
        worst_u = max(worst_u, float(np.max(err_u / bu)))
    return worst_c, worst_u


def test_sample_covers_the_domain(samples):
    n = sum(len(p) for _, p in samples)
    assert n > 900_000
    allp = np.concatenate([p for _, p in samples])
    _, ux, uy, _ = R.macroscopic(allp.astype(np.float64))
    assert np.hypot(ux, uy).max() > 1.4
    assert (allp < 0).any(axis=1).mean() > 0.2


def test_bound_is_sound(samples):
    worst_c, worst_u = ratios(samples)
    print("largest error / bound: lattice %.3f, |u| %.3f" % (worst_c, worst_u))
    assert worst_c < 1.0
    assert worst_u < 1.0
    # and not vacuous: the unperturbed restatement comes within a factor 20 of it
    assert worst_c > 0.05 and worst_u > 0.05


@pytest.mark.parametrize("perturb", ["ow0", "ow1", "ow2", "f45", "m15", "swap", "usq"])
def test_bound_is_tight(samples, perturb):
    worst_c, worst_u = ratios(samples, perturb)
    print("%s: largest error / bound: lattice %.2f, |u| %.2f" % (perturb, worst_c, worst_u))
    assert worst_c > 1.0


def test_emulation_without_perturbation_is_deterministic_and_finite(samples):
    omega, p = samples[0]
    a, ua = R.collide_fast_emulated(p, np.float32(omega))
    b, ub = R.collide_fast_emulated(p, np.float32(omega))
    assert np.array_equal(a, b) and np.array_equal(ua, ub)
    assert np.isfinite(a).all() and np.isfinite(ua).all()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_f64_step_is_the_oracle_step(dtype):
    """f64_step's pull directions, accelerate and bounce-back are the oracle's: the float64
    oracle run of the accelerated source (accel 0) agrees to float64 rounding."""
    nx, ny, density, accel, omega = 37, 11, 0.1, 0.005, 1.85
    cells, obst = O.random_lattice(nx, ny, seed=5, density=density, p_obst=0.1, dtype=dtype)
    ref = R.f64_step(cells, obst, density, accel, omega)
    src, _, _ = O.timestep(cells, obst, density, accel, omega)
    om = np.float64(dtype(omega))
    new, _, _ = O.run(src.astype(np.float64), obst, 1, density, 0.0, om)
    got = ref["cells"].astype(np.float64)
    assert np.array_equal(got[obst != 0], new[obst != 0])
    np.testing.assert_allclose(got, new, rtol=1e-13, atol=1e-16)
    b, bu = R.bound(ref["pulled"], om, R.eps_of(dtype), obst=obst)
    assert (b[obst != 0] == 0).all() and (bu[obst != 0] == 0).all()
    assert (b[obst == 0] > 0).all()
