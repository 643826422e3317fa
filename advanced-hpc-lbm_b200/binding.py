"""ctypes binding of liblbm_b200.so (include/lbm_gpu.h) for the tests and bench.py.

This is the thin Python view of the C-ABI a C host links against; it holds no
compute of its own and has no fallback: if the library is missing, or no GPU is
present when a lattice is created, it raises.  The product host program is C
(advanced-hpc-lbm_b200/host/d2q9-bgk.c); this module exists so that pytest and the
benchmark driver can call exactly the same entry points.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# LBM_B200_LIB selects another build of the same ABI (kernel tuning variants, tools/build_variants.py)
LIB_PATH = os.environ.get("LBM_B200_LIB") or os.path.join(HERE, "liblbm_b200.so")

# lbm_gpu_create flags (include/lbm_gpu.h)
STRICT = 1
OBST_BITS = 2
KERNEL_SCALAR = 4
KERNEL_TMA = 8
KERNEL_VEC4 = 16
SYNC_FLAGS = 32
KERNEL_PERSISTENT = 64
POOL = 128
KERNEL_CLUSTER = 256
KERNEL_TB2 = 512
SYNC_EVENTS = 1024
KERNEL_PAIRS = 2048
KERNEL_TB3 = 4096
STORE_F16 = 8192
IPC_DESC_BYTES = 256
# lbm_gpu_coarse_fields formats
FIELDS_F32 = 0
FIELDS_F16 = 1


class LbmError(RuntimeError):
    pass


class Param(C.Structure):
    """lbm_param == the reference's t_param (d2q9-bgk.c:64-73)."""
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("maxIters", C.c_int), ("reynolds_dim", C.c_int),
                ("density", C.c_float), ("accel", C.c_float), ("omega", C.c_float)]


class ParamF64(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("maxIters", C.c_int), ("reynolds_dim", C.c_int),
                ("density", C.c_double), ("accel", C.c_double), ("omega", C.c_double)]


class Info(C.Structure):
    _fields_ = [("nx", C.c_int), ("ny", C.c_int), ("n_gpus", C.c_int), ("is_f64", C.c_int),
                ("kernel", C.c_int), ("pitch", C.c_int),
                ("free_cells", C.c_longlong), ("local_free_cells", C.c_longlong),
                ("local_row0", C.c_longlong), ("local_rows", C.c_longlong),
                ("steps_done", C.c_longlong), ("kernel_launches", C.c_longlong),
                ("last_run_device_ms", C.c_double), ("last_step_kernel_ms", C.c_double),
                ("device_bytes", C.c_size_t)]


# every symbol include/lbm_gpu.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "lbm_gpu_abi_version": (C.c_int, []),
    "lbm_gpu_last_error": (C.c_char_p, []),
    "lbm_gpu_device_count": (C.c_int, []),
    "lbm_gpu_create": (C.c_int, [C.POINTER(Param), _P, _P, C.c_int, _P, C.c_uint, C.POINTER(_P)]),
    "lbm_gpu_create_f64": (C.c_int, [C.POINTER(ParamF64), _P, _P, C.c_int, _P, C.c_uint, C.POINTER(_P)]),
    "lbm_gpu_create_slab": (C.c_int, [C.POINTER(Param), C.c_longlong, C.c_longlong, C.c_int, _P, _P,
                                      C.c_uint, C.POINTER(_P)]),
    "lbm_gpu_ipc_export": (C.c_int, [_P, _P]),
    "lbm_gpu_ipc_connect": (C.c_int, [_P, _P, _P]),
    "lbm_gpu_ipc_connect_all": (C.c_int, [_P, _P, C.c_int]),
    "lbm_gpu_ipc_prepare": (C.c_int, [_P]),
    "lbm_gpu_run": (C.c_int, [_P, C.c_int, _P]),
    "lbm_gpu_run_f64": (C.c_int, [_P, C.c_int, _P]),
    "lbm_gpu_run_sums": (C.c_int, [_P, C.c_int, _P]),
    "lbm_gpu_run_batch": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "lbm_gpu_set_global_free_cells": (C.c_int, [_P, C.c_longlong]),
    "lbm_gpu_download": (C.c_int, [_P, _P]),
    "lbm_gpu_download_rows": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P]),
    "lbm_gpu_final_fields": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P, _P, _P, _P]),
    "lbm_gpu_av_velocity": (C.c_int, [_P, _P]),
    "lbm_gpu_coarse_fields": (C.c_int, [_P, C.c_int, C.c_uint, C.c_longlong, C.c_longlong, _P, _P, _P, _P]),
    "lbm_gpu_download_f64": (C.c_int, [_P, _P]),
    "lbm_gpu_final_fields_f64": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P, _P, _P, _P]),
    "lbm_gpu_av_velocity_f64": (C.c_int, [_P, _P]),
    "lbm_gpu_digest": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "lbm_gpu_obstacle_force": (C.c_int, [_P, C.c_int, _P, _P]),
    "lbm_gpu_upload": (C.c_int, [_P, _P]),
    "lbm_gpu_upload_f64": (C.c_int, [_P, _P]),
    "lbm_gpu_save_rows": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P]),
    "lbm_gpu_load_rows": (C.c_int, [_P, C.c_longlong, C.c_longlong, _P]),
    "lbm_gpu_get_info": (C.c_int, [_P, C.POINTER(Info)]),
    "lbm_gpu_destroy": (None, [_P]),
    "lbm_gpu_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "lbm_gpu_host_free": (None, [_P]),
}

_lib = None


def load_library(path=None):
    """dlopen the C-ABI library and type every exported symbol.  No fallback."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise LbmError("%s not found: build it with `make` or __graft_entry__.build() "
                       "(there is no CPU fallback)" % p)
    lib = C.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise LbmError(load_library().lbm_gpu_last_error().decode())


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def pack_obstacle_bits(obstacles):
    """(ny,nx) 0/1 array -> the LBM_GPU_OBST_BITS layout (uint32 words, LSB first)."""
    m = np.asarray(obstacles) != 0
    ny, nx = m.shape
    wpr = (nx + 31) // 32
    padded = np.zeros((ny, wpr * 32), dtype=np.uint8)
    padded[:, :nx] = m
    bits = np.packbits(padded.reshape(ny, wpr, 32), axis=-1, bitorder="little")
    return np.ascontiguousarray(bits).view(np.uint32).reshape(ny, wpr)


def lattice_checksum(cells, global_row0=0):
    """numpy restatement of the device checksum (csrc/lbm_kernels.cuh, lbm_digest) for an
    AoS lattice (rows, nx, 9) of float32 or float64."""
    cells = np.ascontiguousarray(cells)
    rows, nx, _ = cells.shape
    bits = cells.view(np.uint32 if cells.dtype == np.float32 else np.uint64).astype(np.uint64)
    g = (np.arange(rows, dtype=np.uint64)[:, None] + np.uint64(global_row0)) * np.uint64(nx) \
        + np.arange(nx, dtype=np.uint64)[None, :]
    k = np.arange(1, 10, dtype=np.uint64)
    with np.errstate(over="ignore"):
        w = (g[:, :, None] * np.uint64(0x9E3779B97F4A7C15) + k[None, None, :] * np.uint64(0xC2B2AE3D27D4EB4F)) | np.uint64(1)
        return int(np.sum(bits * w, dtype=np.uint64))


class PinnedArray:
    """numpy view of page-locked host memory from lbm_gpu_host_alloc."""

    def __init__(self, shape, dtype):
        self._lib = load_library()
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _check(self._lib.lbm_gpu_host_alloc(max(n, 1), C.byref(p)))
        self._p = p
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._p is not None:
            self.array = None
            self._lib.lbm_gpu_host_free(self._p)
            self._p = None


class Lattice:
    """One d2q9 lattice on the GPU(s): the replacement of the reference's step loop.

    cells     (ny,nx,9) float32 AoS like t_speed, or None for the rest state
    obstacles (ny,nx) int32 like the reference's array (or packed bits with bits=True)
    """

    def __init__(self, nx, ny, density, accel, omega, cells=None, obstacles=None, n_gpus=1,
                 device_ids=None, flags=0, f64=False, reynolds_dim=10, max_iters=0, bits=False,
                 slab=None):
        self.lib = load_library()
        self.f64 = bool(f64)
        self.nx, self.ny = int(nx), int(ny)
        self.dtype = np.float64 if f64 else np.float32
        self.h = C.c_void_p()
        if bits:
            flags |= OBST_BITS
        rows = self.ny if slab is None else int(slab[1])
        if cells is not None:
            cells = np.ascontiguousarray(cells, dtype=self.dtype)
            assert cells.size == rows * self.nx * 9
        if obstacles is not None:
            if bits:
                obstacles = np.ascontiguousarray(obstacles, dtype=np.uint32)
                assert obstacles.size == rows * ((self.nx + 31) // 32)
            else:
                obstacles = np.ascontiguousarray(obstacles, dtype=np.int32)
                assert obstacles.size == rows * self.nx
        self.rows = rows
        self.row0 = 0 if slab is None else int(slab[0])
        self.f16 = bool(flags & STORE_F16)
        dev = None
        if device_ids is not None:
            dev = np.ascontiguousarray(device_ids, dtype=np.int32)
        if f64:
            assert slab is None
            p = ParamF64(self.nx, self.ny, int(max_iters), int(reynolds_dim), density, accel, omega)
            _check(self.lib.lbm_gpu_create_f64(C.byref(p), _ptr(cells), _ptr(obstacles), int(n_gpus),
                                               _ptr(dev), flags, C.byref(self.h)))
        elif slab is None:
            p = Param(self.nx, self.ny, int(max_iters), int(reynolds_dim), density, accel, omega)
            _check(self.lib.lbm_gpu_create(C.byref(p), _ptr(cells), _ptr(obstacles), int(n_gpus),
                                           _ptr(dev), flags, C.byref(self.h)))
        else:
            p = Param(self.nx, self.ny, int(max_iters), int(reynolds_dim), density, accel, omega)
            device = 0 if device_ids is None else int(device_ids[0])
            _check(self.lib.lbm_gpu_create_slab(C.byref(p), self.row0, rows, device, _ptr(cells),
                                                _ptr(obstacles), flags, C.byref(self.h)))

    # -- multi-process wiring -------------------------------------------------------
    def ipc_export(self):
        buf = np.zeros(IPC_DESC_BYTES, dtype=np.uint8)
        _check(self.lib.lbm_gpu_ipc_export(self.h, _ptr(buf)))
        return buf

    def ipc_connect(self, desc_below, desc_above):
        b = np.ascontiguousarray(desc_below, dtype=np.uint8)
        a = np.ascontiguousarray(desc_above, dtype=np.uint8)
        _check(self.lib.lbm_gpu_ipc_connect(self.h, _ptr(b), _ptr(a)))

    def ipc_connect_all(self, descs):
        """descs: (world, IPC_DESC_BYTES) uint8, the descriptors of ALL ranks in any order."""
        d = np.ascontiguousarray(descs, dtype=np.uint8).reshape(-1, IPC_DESC_BYTES)
        _check(self.lib.lbm_gpu_ipc_connect_all(self.h, _ptr(d), int(d.shape[0])))

    def ipc_prepare(self):
        _check(self.lib.lbm_gpu_ipc_prepare(self.h))

    def set_global_free_cells(self, n):
        _check(self.lib.lbm_gpu_set_global_free_cells(self.h, int(n)))

    # -- the step loop ----------------------------------------------------------------
    def run(self, n_steps, out=None):
        """n_steps timesteps; returns the av_vels array (one value per step)."""
        av = out if out is not None else np.empty(max(n_steps, 0), dtype=self.dtype)
        fn = self.lib.lbm_gpu_run_f64 if self.f64 else self.lib.lbm_gpu_run
        _check(fn(self.h, int(n_steps), _ptr(av)))
        return av

    def run_sums(self, n_steps):
        s = np.empty(max(n_steps, 0), dtype=np.float64)
        _check(self.lib.lbm_gpu_run_sums(self.h, int(n_steps), _ptr(s)))
        return s

    def run_timed(self, n_steps):
        """n_steps without fetching av_vels; returns device milliseconds (CUDA events)."""
        fn = self.lib.lbm_gpu_run_f64 if self.f64 else self.lib.lbm_gpu_run
        _check(fn(self.h, int(n_steps), None))
        return self.info().last_run_device_ms

    # -- results --------------------------------------------------------------------
    def download(self, out=None):
        cells = out if out is not None else np.empty((self.rows, self.nx, 9), dtype=self.dtype)
        fn = self.lib.lbm_gpu_download_f64 if self.f64 else self.lib.lbm_gpu_download
        _check(fn(self.h, _ptr(cells)))
        return cells

    def download_rows(self, row0, nrows):
        cells = np.empty((nrows, self.nx, 9), dtype=np.float32)
        _check(self.lib.lbm_gpu_download_rows(self.h, int(row0), int(nrows), _ptr(cells)))
        return cells

    def upload(self, cells):
        cells = np.ascontiguousarray(cells, dtype=self.dtype)
        assert cells.size == self.rows * self.nx * 9
        fn = self.lib.lbm_gpu_upload_f64 if self.f64 else self.lib.lbm_gpu_upload
        _check(fn(self.h, _ptr(cells)))

    @property
    def record_dtype(self):
        """Element type of save_rows / load_rows: the handle's stored type (binary16 as uint16 bits)."""
        return np.float64 if self.f64 else (np.uint16 if self.f16 else np.float32)

    def save_rows(self, row0=None, nrows=None):
        """Rows [row0, row0 + nrows) of the stored lattice, (nrows, nx, 9) of record_dtype, bit for bit
        (lbm_gpu_save_rows).  By default every row this handle holds."""
        row0 = self.row0 if row0 is None else int(row0)
        nrows = self.row0 + self.rows - row0 if nrows is None else int(nrows)
        out = np.empty((max(nrows, 0), self.nx, 9), dtype=self.record_dtype)
        _check(self.lib.lbm_gpu_save_rows(self.h, row0, nrows, _ptr(out)))
        return out

    def load_rows(self, row0, arr):
        """Put rows saved by save_rows back from row0 on (lbm_gpu_load_rows).  A slab handle that holds
        part of the grid must pass barrier / ipc_prepare / barrier with the other ranks before it runs."""
        arr = np.asarray(arr)
        if arr.dtype != self.record_dtype:
            raise LbmError("load_rows: records of this lattice are %s, got %s" % (np.dtype(self.record_dtype), arr.dtype))
        if arr.ndim != 3 or arr.shape[1:] != (self.nx, 9):
            raise LbmError("load_rows: need shape (nrows, %d, 9), got %s" % (self.nx, arr.shape))
        arr = np.ascontiguousarray(arr)
        _check(self.lib.lbm_gpu_load_rows(self.h, int(row0), arr.shape[0], _ptr(arr)))

    def final_fields(self, row0=None, nrows=None, out=None):
        """(u_x, u_y, |u|, pressure) as write_values computes them (d2q9-bgk.c:2937-2976)."""
        row0 = self.row0 if row0 is None else row0
        nrows = self.rows if nrows is None else nrows
        if out is None:
            out = [np.empty((nrows, self.nx), dtype=self.dtype) for _ in range(4)]
        fn = self.lib.lbm_gpu_final_fields_f64 if self.f64 else self.lib.lbm_gpu_final_fields
        _check(fn(self.h, int(row0), int(nrows), *[_ptr(o) for o in out]))
        return tuple(out)

    def coarse_rows(self, factor):
        """(crow0, ncrows): the coarse rows of `factor` whose fine rows this handle holds entirely."""
        ncy = -(-self.ny // factor)
        end = self.row0 + self.rows
        first = -(-self.row0 // factor)
        last = ncy if end == self.ny else end // factor
        return first, max(0, last - first)

    def coarse_fields(self, factor, f16=False, crow0=None, ncrows=None, out=None):
        """Block means over factor x factor cells of (u_x, u_y, |u|, pressure), computed on the GPU
        (lbm_gpu_coarse_fields): four arrays of shape (ncrows, ceil(nx / factor)), float32, or with
        f16 float16 holding the pressure shifted by p0 = float32(density) * float32(1/3) (decode
        it as float32(h) + p0).  By default every coarse row this handle holds entirely."""
        d0, dn = self.coarse_rows(factor)
        crow0 = d0 if crow0 is None else crow0
        ncrows = dn if ncrows is None else ncrows
        if out is None:
            ncx = -(-self.nx // factor)
            out = [np.empty((max(ncrows, 0), ncx), dtype=np.float16 if f16 else np.float32) for _ in range(4)]
        _check(self.lib.lbm_gpu_coarse_fields(self.h, int(factor), FIELDS_F16 if f16 else FIELDS_F32, int(crow0),
                                              int(ncrows), *[_ptr(o) for o in out]))
        return tuple(out)

    def av_velocity(self):
        if self.f64:
            v = C.c_double()
            _check(self.lib.lbm_gpu_av_velocity_f64(self.h, C.byref(v)))
        else:
            v = C.c_float()
            _check(self.lib.lbm_gpu_av_velocity(self.h, C.byref(v)))
        return v.value

    def digest(self):
        """(total_density, checksum) of the local rows: exact, additive over ranks."""
        d, c = C.c_double(), C.c_ulonglong()
        _check(self.lib.lbm_gpu_digest(self.h, C.byref(d), C.byref(c)))
        return d.value, c.value

    def obstacle_force(self, boxes=None):
        """Momentum-exchange force (fx, fy) on the solid cells of each box, computed on the GPU
        (lbm_gpu_obstacle_force): float64 array of shape (n, 2).  boxes: (n, 4) ints {x0, y0, x1, y1},
        half-open global cell ranges; None is the whole grid.  A slab handle returns its rows' share."""
        if boxes is None:
            out = np.empty((1, 2), dtype=np.float64)
            _check(self.lib.lbm_gpu_obstacle_force(self.h, 1, None, _ptr(out)))
            return out
        b = np.ascontiguousarray(boxes, dtype=np.int32).reshape(-1, 4)
        out = np.empty((b.shape[0], 2), dtype=np.float64)
        _check(self.lib.lbm_gpu_obstacle_force(self.h, b.shape[0], _ptr(b), _ptr(out)))
        return out

    def info(self):
        i = Info()
        _check(self.lib.lbm_gpu_get_info(self.h, C.byref(i)))
        return i

    def close(self):
        if self.h:
            self.lib.lbm_gpu_destroy(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def run_batch(lattices, n_steps):
    """Advance every Lattice of `lattices` by n_steps in one batch on the GPU (parameter
    sweeps; lbm_gpu_run_batch).  Returns the av_vels of each, shape (n, n_steps) float32:
    the same bits as lat.run(n_steps) on each in turn."""
    lib = load_library()
    lattices = list(lattices)
    handles = (C.c_void_p * max(len(lattices), 1))(*[lat.h.value for lat in lattices])
    av = np.empty((len(lattices), max(int(n_steps), 0)), dtype=np.float32)
    _check(lib.lbm_gpu_run_batch(C.cast(handles, C.c_void_p), len(lattices), int(n_steps), _ptr(av)))
    return av
