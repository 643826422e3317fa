"""Exact CPU restatement of lbm_gpu_coarse_fields (block means of the per-cell fields) in
numpy integers, from the per-cell values of final_fields.  TEST INFRASTRUCTURE ONLY."""
import numpy as np

FIX_BITS = 32            # each cell value enters its block's sum as rint(v * 2^32)
LIMIT = 2.0 ** 15        # a value that is not finite or of this magnitude makes its block NaN


def p0(density):
    """The obstacle pressure of final_fields, float32(density) * float32(1/3): the shift of
    the binary16 pressure."""
    return np.float32(np.float32(density) * (np.float32(1) / np.float32(3)))


def block_sums(v, factor):
    """(S, bad) per factor x factor block of the (rows, nx) float32 array v: S the int64 sum of
    rint(float64(v) * 2^32) over the block's cells, bad whether any of them is not finite or
    of magnitude LIMIT or more (it then adds nothing).  Blocks at the right and bottom are
    smaller."""
    ny, nx = v.shape
    ncy, ncx = -(-ny // factor), -(-nx // factor)
    x = np.asarray(v, dtype=np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        bad = ~(np.abs(x) < LIMIT)
    q = np.where(bad, 0.0, np.rint(np.ldexp(np.where(bad, 0.0, x), FIX_BITS))).astype(np.int64)
    pq = np.zeros((ncy * factor, ncx * factor), dtype=np.int64)
    pb = np.zeros(pq.shape, dtype=bool)
    pq[:ny, :nx] = q
    pb[:ny, :nx] = bad
    S = pq.reshape(ncy, factor, ncx, factor).sum(axis=(1, 3), dtype=np.int64)   # |S| < 2^63
    B = pb.reshape(ncy, factor, ncx, factor).any(axis=(1, 3))
    return S, B


def block_cells(ny, nx, factor):
    """Number of cells of each block."""
    rows = np.minimum(factor, ny - np.arange(0, ny, factor))
    cols = np.minimum(factor, nx - np.arange(0, nx, factor))
    return rows[:, None].astype(np.int64) * cols[None, :]


def mean(S, B, cells):
    """(float32)((double)S * 2^-32 / cells), NaN where B."""
    m = (S.astype(np.float64) * 2.0 ** -FIX_BITS / cells.astype(np.float64)).astype(np.float32)
    m[B] = np.nan
    return m


def to_f16(fields, density):
    """The binary16 outputs from fp32 values: u_x, u_y, |u| rounded, pressure shifted by p0 in
    fp32 and then rounded."""
    ux, uy, u, p = fields
    with np.errstate(invalid="ignore", over="ignore"):
        return (ux.astype(np.float16), uy.astype(np.float16), u.astype(np.float16),
                (p - p0(density)).astype(np.float16))


def coarse_fields(fields, factor, density, f16=False):
    """What lbm_gpu_coarse_fields returns for the whole grid whose per-cell fields (u_x, u_y,
    |u|, pressure; float32, shape (ny, nx)) are `fields`.  factor 1 with f16 converts each
    cell's values directly; factor 1 in fp32 is the fields themselves."""
    fields = [np.asarray(f, dtype=np.float32) for f in fields]
    if factor == 1:
        out = tuple(f.copy() for f in fields)
    else:
        ny, nx = fields[0].shape
        cells = block_cells(ny, nx, factor)
        out = tuple(mean(*block_sums(f, factor), cells) for f in fields)
    return to_f16(out, density) if f16 else out


def decode_pressure(h, density):
    """The user's decoding of the binary16 pressure."""
    return h.astype(np.float32) + p0(density)
