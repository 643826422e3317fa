"""CPU reference of shifted binary16 lattice storage (LBM_GPU_STORE_F16): the fp32 oracle of
oracle_lib, one timestep at a time, with the lattice encoded and decoded by numpy between
steps.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

import oracle_lib as O


def rest_shift(density):
    """The fp32 rest-state values of the nine speeds, computed as oracle_init_cells does."""
    d = np.float32(density)
    w0, w1, w2 = d * np.float32(4) / np.float32(9), d / np.float32(9), d / np.float32(36)
    return np.array([w0] + [w1] * 4 + [w2] * 4, dtype=np.float32)


def f16_encode(cells, density):
    """Shifted binary16 storage: one fp32 subtract, then round to nearest even."""
    return (np.asarray(cells, dtype=np.float32) - rest_shift(density)).astype(np.float16)


def f16_decode(stored, density):
    return stored.astype(np.float32) + rest_shift(density)


def run_f16(cells, obstacles, iters, density, accel, omega):
    """The fp32 oracle one step at a time with the lattice stored as shifted binary16 between
    steps.  Returns (final decoded cells, av_vels with double accumulation)."""
    state = f16_encode(cells, density)
    obst = np.ascontiguousarray(obstacles, dtype=np.int32)
    avd = np.empty(iters, dtype=np.float64)
    for t in range(iters):
        new, _, av = O.run(f16_decode(state, density), obst, 1, density, accel, omega)
        avd[t] = av[0]
        state = f16_encode(new, density)
    return f16_decode(state, density), avd
