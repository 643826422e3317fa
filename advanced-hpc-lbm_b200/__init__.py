"""advanced-hpc-lbm_b200: the d2q9-bgk timestep loop for NVIDIA B200 (sm_100a).

The product is a C-ABI shared library (csrc/ -> liblbm_b200.so, declared in
include/lbm_gpu.h) plus a C host program with the reference's command line
(host/d2q9-bgk.c).  This Python package is only the ctypes view of that ABI used by
the tests and the benchmark driver.  The directory name contains hyphens, so import
it with importlib.import_module("advanced-hpc-lbm_b200") or through the root-level
shim `lbm_b200`.
"""
from .binding import (FIELDS_F16, FIELDS_F32, IPC_DESC_BYTES, KERNEL_CLUSTER, KERNEL_PAIRS, KERNEL_PERSISTENT, KERNEL_SCALAR, KERNEL_TB2, KERNEL_TB3, KERNEL_TMA, KERNEL_VEC4, LIB_PATH, OBST_BITS, POOL, STORE_F16, STRICT,
                      SYNC_EVENTS, SYNC_FLAGS,
                      SYMBOLS, Info, Lattice, LbmError, Param, ParamF64, PinnedArray, lattice_checksum, load_library,
                      pack_obstacle_bits, run_batch)
from .slabs import split_rows, ring_neighbours

__all__ = ["FIELDS_F16", "FIELDS_F32", "IPC_DESC_BYTES", "KERNEL_CLUSTER", "KERNEL_PAIRS", "KERNEL_PERSISTENT", "KERNEL_SCALAR", "KERNEL_TB2", "KERNEL_TB3", "KERNEL_TMA", "KERNEL_VEC4", "LIB_PATH", "OBST_BITS", "POOL", "STORE_F16", "STRICT",
           "SYNC_EVENTS", "SYNC_FLAGS",
           "SYMBOLS", "Info", "Lattice", "LbmError", "Param", "ParamF64", "PinnedArray", "lattice_checksum", "load_library",
           "pack_obstacle_bits", "run_batch", "split_rows", "ring_neighbours"]
