"""Overlapped K10 passes (a block of pass p+1 waits for its nine neighbour tiles of pass p, not
for the whole grid) against passes that do not overlap (LBM_GPU_NO_TB3_OVERLAP=1): the same
lattice and the same per-step sums, on grids with one, two, three and many strips and segments
(the neighbour list wraps onto itself), ragged widths and heights, every kind of pass that can
follow K10, split runs, an upload between runs and a cell that turns NaN.
"""
import numpy as np
import pytest

import lbm_b200 as L
import oracle_lib as O

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85


@pytest.fixture
def make(monkeypatch):
    """make(overlap, nx, ny, seg_rows, cells, obst) -> a K10 lattice; the switches are read at creation"""
    def create(overlap, nx, ny, seg_rows, cells, obst):
        if overlap:
            monkeypatch.delenv("LBM_GPU_NO_TB3_OVERLAP", raising=False)
        else:
            monkeypatch.setenv("LBM_GPU_NO_TB3_OVERLAP", "1")
        monkeypatch.setenv("LBM_TB3_SEG_ROWS", str(seg_rows))
        lat = L.Lattice(nx, ny, D, A, W, cells=cells, obstacles=obst, flags=L.KERNEL_TB3)
        assert lat.info().kernel == L.KERNEL_TB3
        return lat
    return create


def both(make, nx, ny, seg_rows, cells, obst, runs, upload=None):
    """digest and concatenated per-step sums of the run sequence `runs`, overlap on and off"""
    res = []
    for overlap in (True, False):
        with make(overlap, nx, ny, seg_rows, cells, obst) as lat:
            av = []
            for i, n in enumerate(runs):
                if upload is not None and i == len(runs) // 2:
                    lat.upload(upload)
                av.append(lat.run(n))
            res.append((lat.digest(), np.concatenate(av)))
    return res


# nx: one narrow strip (the span wraps onto itself), two, three (ragged), eleven with a last strip
# narrower than the others; seg_rows over ny: one, two, three and many segments, the last one shorter
@pytest.mark.parametrize("nx", [128, 512, 1028, 4100])
@pytest.mark.parametrize("ny,seg_rows", [(24, 24), (26, 13), (26, 9), (61, 8), (40, 3)])
def test_strips_and_segments(make, nx, ny, seg_rows):
    cells, obst = O.random_lattice(nx, ny, seed=nx + ny, p_obst=0.02)
    on, off = both(make, nx, ny, seg_rows, cells, obst, [13])
    assert on[0] == off[0]
    assert np.array_equal(on[1], off[1]) and np.all(np.isfinite(on[1]))


@pytest.mark.parametrize("steps", [3, 4, 5, 6, 200])
def test_run_lengths(make, steps):
    """3k+1 and 3k+2 timesteps end with K1a and K7 after overlapped K10 passes"""
    nx, ny = 1028, 48
    cells, obst = O.random_lattice(nx, ny, seed=steps, p_obst=0.02)
    on, off = both(make, nx, ny, 8, cells, obst, [steps])
    assert on[0] == off[0]
    assert np.array_equal(on[1], off[1]) and np.all(np.isfinite(on[1]))


def test_split_runs_equal_one_run(make):
    nx, ny = 1028, 40
    cells, obst = O.random_lattice(nx, ny, seed=5, p_obst=0.02)
    one = both(make, nx, ny, 8, cells, obst, [31])
    parts = both(make, nx, ny, 8, cells, obst, [7, 1, 9, 0, 2, 12])
    for r in one + parts:
        assert r[0] == one[0][0]
        assert np.array_equal(r[1], one[0][1])


def test_upload_between_runs(make):
    nx, ny = 512, 30
    cells, obst = O.random_lattice(nx, ny, seed=6, p_obst=0.02)
    other, _ = O.random_lattice(nx, ny, seed=7)
    on, off = both(make, nx, ny, 5, cells, obst, [10, 12], upload=other)
    assert on[0] == off[0]
    assert np.array_equal(on[1], off[1])
    # the upload replaced the state: the second run is that of `other` alone
    fresh = both(make, nx, ny, 5, other, obst, [12])
    assert fresh[0][0] == on[0]
    assert np.array_equal(fresh[0][1], on[1][10:])


def test_nan_cell_reads_nan(make):
    nx, ny = 512, 30
    cells, obst = O.random_lattice(nx, ny, seed=2, p_obst=0.0, walls=False)
    cells[14:17, 99:102, :] = 0.0          # a hole of zero density: cell (15,100) pulls only zeros, u = 0/0
    for overlap in (True, False):
        with make(overlap, nx, ny, 5, cells, obst) as lat:
            av = lat.run(9)
        assert np.isnan(av).all(), av
