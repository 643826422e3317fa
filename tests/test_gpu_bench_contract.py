"""bench.py's GPU arm on a reduced grid (LBM_BENCH_NX / LBM_BENCH_ROWS): the JSON line
carries every key of the benchmark contract and the numbers are self-consistent."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_gpu_arm_prints_contract_line():
    env = dict(os.environ, LBM_BENCH_NX="4096", LBM_BENCH_ROWS="4096", LBM_BENCH_CPU_BUDGET_S="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3",
                        "--timesteps", "20", "--no-cpu-baseline"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["unit"] == "MLUPS" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3
    assert d["scaling"] == "weak" and d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["kernel_variant"] == 512 and d["gpu_launches"] == 2 * 20 // 2   # two timesteps per kernel launch (K7)
    cells = 4096 * 4096
    assert abs(d["value"] - cells * 20 * 2 / (d["ms_per_step"] * 2 * 1e-3) / 1e6) < 1e-6 * d["value"]
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    assert rf["timesteps_per_launch"] == 2 and rf["algorithmic_bytes_per_update"] == 36.0
    assert abs(rf["achieved"] - d["value"] * 36e-3) < 1e-6 * rf["achieved"]
    assert 0.3 < rf["frac"] < 1.3
    assert "traffic_source" in rf and len(rf["library_sha256_16"]) == 16
    par = d["parity"]
    assert par["checked"] and par["ok"] and all(c["strict_lattice_equals_oracle"] for c in par["cases"])
    assert par["mass_conservation_full_grid"]["ok"]
    assert d["strong"]["value"] == d["value"]
    sh = d["shipped"]
    assert set(sh) == {"128x128", "128x256", "256x256", "1024x1024"} and all(v["check"] == "pass" for v in sh.values())
    e = d["e2e"]
    assert e["unit"] == "MLUPS" and 0 < e["value"] < d["value"]
    assert e["h2d_bytes_per_step"] == cells * 4 and e["d2h_bytes_per_step"] == 4 * cells * 4 + 20 * 4
    assert d["config"]["workload"].startswith("synthetic 4096x4096 channel")
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def test_dump_outputs_is_reproducible_and_follows_steps(tmp_path):
    """--dump-outputs: the arrays are those of the last timed step (rebuilt here with a fresh
    lattice); the same arguments give the same arrays; one more timed step gives others."""
    import numpy as np
    import lbm_b200 as L
    from tools.make_inputs import channel_mask
    nx, ny, T, warmup = 4096, 2048, 20, 3
    env = dict(os.environ, LBM_BENCH_NX=str(nx), LBM_BENCH_ROWS=str(ny))

    def dump(name, steps):
        d = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                            "--timesteps", str(T), "--dump-outputs", str(d), "--no-cpu-baseline", "--no-e2e",
                            "--no-parity", "--no-shipped", "--no-strong"],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        assert all(p.suffix == ".npy" for p in d.iterdir())
        return {p.stem: np.load(p) for p in d.iterdir()}

    a, b, c = dump("a", 2), dump("b", 2), dump("c", 3)
    assert set(a) == {"av_vels", "cells_rows", "cells_rows_index"}
    assert a["av_vels"].shape == (T,) and a["cells_rows"].shape == (64, nx, 9)
    # the same workload from scratch: warm-up plus timed steps of T timesteps, the last one fetched
    with L.Lattice(nx, ny, 0.1, 0.005, 1.85, obstacles=channel_mask(nx, ny)) as lat:
        for _ in range(warmup + 2 - 1):
            lat.run_timed(T)
        av = (lat.run_sums(T) / lat.info().local_free_cells).astype(np.float32)
        rows = np.stack([lat.download_rows(int(r), 1)[0] for r in a["cells_rows_index"]])
    assert np.array_equal(a["av_vels"], av)
    assert np.array_equal(a["cells_rows"], rows)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.all(a["av_vels"] > 0) and np.isfinite(a["cells_rows"]).all()
    assert (np.abs(a["cells_rows"]).sum(axis=(1, 2)) > 0).all()        # every sampled row was filled in
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["cells_rows_index"], c["cells_rows_index"])
    assert not np.array_equal(a["cells_rows"], c["cells_rows"])
    assert not np.array_equal(a["av_vels"], c["av_vels"])
