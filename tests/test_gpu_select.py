"""Which kernel runs a lattice: one table of flags, shapes and layouts against the kernel that
lbm_gpu_get_info reports, or the refusal.

Sizes stay far from the device-dependent boundaries (L2 size, waves of blocks, resident
blocks), so the table holds on any B200.  Slab handles are wired to themselves: a slab that
holds the whole grid may name its own window as both neighbours, a ring of one process.
"""
import re

import pytest

import lbm_b200 as L

pytestmark = pytest.mark.gpu
D, A, W = 0.1, 0.005, 1.85
F16 = L.STORE_F16


def case(tag, nx, ny, expect, **kw):
    """expect: the kernel, a substring of the refusal, or for a slab handle wired into a ring
    (kw connect="all" or "pair") (kernel at create, kernel after connect, step launches of run(6))"""
    return pytest.param(nx, ny, kw, expect, id=tag)


def slab(ny, rows=None):
    return dict(slab=(0, ny if rows is None else rows), device_ids=[0])


CASES = [
    # defaults
    case("default-128x128", 128, 128, L.KERNEL_PAIRS),
    case("default-640x512", 640, 512, L.KERNEL_PERSISTENT),
    case("default-130x16", 130, 16, L.KERNEL_PERSISTENT),
    case("default-4098x4096", 4098, 4096, L.KERNEL_VEC4),
    case("default-4096x4096", 4096, 4096, L.KERNEL_TB2),
    case("default-16384x4096", 16384, 4096, L.KERNEL_TB3),
    case("f64-128x128", 128, 128, L.KERNEL_PERSISTENT, f64=True),
    case("f64-4096x4096", 4096, 4096, L.KERNEL_VEC4, f64=True),
    case("2slabs-128x128", 128, 128, L.KERNEL_TB2, n_gpus=2, device_ids=[0, 0]),
    case("2slabs-4098x4096", 4098, 4096, L.KERNEL_VEC4, n_gpus=2, device_ids=[0, 0]),
    case("2slabs-16384x4096", 16384, 4096, L.KERNEL_TB2, n_gpus=2, device_ids=[0, 0]),
    case("f16-64x32", 64, 32, L.KERNEL_TB2, flags=F16),
    case("f16-68x32", 68, 32, L.KERNEL_VEC4, flags=F16),
    # every forced kernel, where it applies and where it is refused
    case("SCALAR", 130, 64, L.KERNEL_SCALAR, flags=L.KERNEL_SCALAR),
    case("SCALAR-f16", 64, 32, "VEC4 or LBM_GPU_KERNEL_TB2 only", flags=F16 | L.KERNEL_SCALAR),
    case("TMA", 1100, 40, L.KERNEL_TMA, flags=L.KERNEL_TMA),
    case("TMA-f64", 1100, 40, "single precision only", flags=L.KERNEL_TMA, f64=True),
    case("VEC4", 4096, 4096, L.KERNEL_VEC4, flags=L.KERNEL_VEC4),
    case("VEC4-f16", 64, 32, L.KERNEL_VEC4, flags=F16 | L.KERNEL_VEC4),
    case("PERSISTENT", 1024, 600, L.KERNEL_PERSISTENT, flags=L.KERNEL_PERSISTENT),
    case("PERSISTENT-2slabs", 1024, 600, "persistent kernel handles a single slab only", flags=L.KERNEL_PERSISTENT,
         n_gpus=2, device_ids=[0, 0]),
    case("CLUSTER", 128, 128, L.KERNEL_CLUSTER, flags=L.KERNEL_CLUSTER),
    case("CLUSTER-2048x2048", 2048, 2048, "fits in one cluster", flags=L.KERNEL_CLUSTER),
    case("PAIRS", 256, 256, L.KERNEL_PAIRS, flags=L.KERNEL_PAIRS),
    case("PAIRS-512x64", 512, 64, "pairs kernel", flags=L.KERNEL_PAIRS),
    case("TB2", 16384, 4096, L.KERNEL_TB2, flags=L.KERNEL_TB2),
    case("TB2-130x64", 130, 64, "two-step kernel", flags=L.KERNEL_TB2),
    case("TB2-f16", 64, 32, L.KERNEL_TB2, flags=F16 | L.KERNEL_TB2),
    case("TB2-f16-68x32", 68, 32, "multiple of 8", flags=F16 | L.KERNEL_TB2),
    case("TB3", 512, 40, L.KERNEL_TB3, flags=L.KERNEL_TB3),
    case("TB3-2slabs", 512, 40, "three-step kernel", flags=L.KERNEL_TB3, n_gpus=2, device_ids=[0, 0]),
    case("f16-f64", 64, 32, "fp32 lattices only", flags=F16, f64=True),
    case("f16-2slabs", 64, 32, "n_gpus == 1", flags=F16, n_gpus=2, device_ids=[0, 0]),
    case("f16-slab", 64, 32, "not slab handles", flags=F16, **slab(32)),
    # two kernel flags are refused, whichever they are
    case("TB2|TB3", 16384, 4096, "more than one kernel", flags=L.KERNEL_TB2 | L.KERNEL_TB3),
    case("PAIRS|TMA", 128, 128, "more than one kernel", flags=L.KERNEL_PAIRS | L.KERNEL_TMA),
    case("SCALAR|VEC4", 4096, 64, "more than one kernel", flags=L.KERNEL_SCALAR | L.KERNEL_VEC4),
    case("f16-VEC4|TB2", 64, 32, "more than one kernel", flags=F16 | L.KERNEL_VEC4 | L.KERNEL_TB2),
    # slab handles (lbm_gpu_create_slab)
    case("slab-partial", 512, 64, L.KERNEL_VEC4, **slab(64, 32)),
    case("slab-partial-TB2", 512, 64, L.KERNEL_VEC4, flags=L.KERNEL_TB2, **slab(64, 32)),   # K7 is decided at connect
    case("slab-whole", 16384, 4096, L.KERNEL_TB3, **slab(4096)),
    case("slab-PERSISTENT", 128, 128, "persistent kernel handles a single slab only", flags=L.KERNEL_PERSISTENT, **slab(128)),
    case("slab-CLUSTER", 128, 128, "fits in one cluster", flags=L.KERNEL_CLUSTER, **slab(128)),
    case("slab-PAIRS", 128, 128, "pairs kernel", flags=L.KERNEL_PAIRS, **slab(128)),
    case("slab-partial-TB3", 512, 64, "three-step kernel", flags=L.KERNEL_TB3, **slab(64, 32)),
    # a whole-grid slab handle in a ring of one process: K7 with connect_all, K1a otherwise
    case("ring-all-16384x4096", 16384, 4096, (L.KERNEL_TB3, L.KERNEL_TB2, 3), connect="all", **slab(4096)),
    case("ring-pair-16384x4096", 16384, 4096, (L.KERNEL_TB3, L.KERNEL_VEC4, 6), connect="pair", **slab(4096)),
    case("ring-pair-4096x4096", 4096, 4096, (L.KERNEL_TB2, L.KERNEL_VEC4, 6), connect="pair", **slab(4096)),
    case("ring-all-TB3", 512, 40, "three-step kernel", flags=L.KERNEL_TB3, connect="all", **slab(40)),
]


@pytest.mark.parametrize("nx,ny,kw,expect", CASES)
def test_selection(nx, ny, kw, expect):
    kw = dict(kw)
    connect = kw.pop("connect", None)

    def create_and_connect():
        lat = L.Lattice(nx, ny, D, A, W, **kw)
        created = lat.info().kernel
        try:
            if connect:
                desc = lat.ipc_export()
                if connect == "all":
                    lat.ipc_connect_all(desc[None])
                else:
                    lat.ipc_connect(desc, desc)
                lat.ipc_prepare()
        except L.LbmError:
            lat.close()
            raise
        return lat, created

    if isinstance(expect, str):
        with pytest.raises(L.LbmError, match=re.escape(expect)):
            create_and_connect()[0].close()
        return
    lat, created = create_and_connect()
    with lat:
        if not connect:
            assert created == expect
            return
        at_create, after, step_launches = expect
        assert (created, lat.info().kernel) == (at_create, after)
        before = lat.info().kernel_launches
        lat.run(6)
        # besides the step kernels, a ring's run ends with one wait for the neighbours and one
        # compaction of the per-step sums
        assert lat.info().kernel_launches - before == step_launches + 2
