"""Accuracy of shifted binary16 lattice storage (LBM_GPU_STORE_F16) on the shipped inputs, on
the CPU: tests/oracle_f16.run_f16 (the fp32 oracle with the lattice encoded between steps) over
the full step count, against the fp64 golden files with check.py's criterion (largest
|percentage difference| of av_vels and of the final pressure).  The plain fp32 oracle runs
alongside as the baseline.

    python tools/f16_accuracy.py 128x128 [128x256 256x256]      (one line of JSON per input)
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_f16 as H  # noqa: E402
import oracle_lib as O  # noqa: E402
from tools.make_inputs import SHIPPED, shipped_mask  # noqa: E402


def worst_pct(ref, sim):
    delta = ref - sim
    with np.errstate(divide="ignore", invalid="ignore"):
        pct = 100.0 * (delta / (ref - delta))
    return float(np.max(np.abs(pct)))


def main(names):
    for name in names:
        nx, ny, iters, _re, rho, acc, om, _r, _c = SHIPPED[name]
        obst = shipped_mask(name).astype(np.int32)
        g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        cells = O.rest_cells(nx, ny, rho, np.float32)
        rho, acc, om = np.float32(rho), np.float32(acc), np.float32(om)
        t0 = time.time()
        res = {"input": name, "steps": iters}
        fin32, _, av32 = O.run(cells, obst, iters, rho, acc, om)
        fin16, av16 = H.run_f16(cells, obst, iters, rho, acc, om)
        for tag, fin, av in (("f32", fin32, av32), ("f16", fin16, av16)):
            p = O.final_state(fin, obst, rho)[3]
            res[tag + "_av_vels_pct"] = worst_pct(g["av_vels"], av.astype(np.float64))
            res[tag + "_pressure_pct"] = worst_pct(g["pressure"].ravel(), p.astype(np.float64).ravel())
        res["f16_passes_1pct"] = bool(res["f16_av_vels_pct"] <= 1.0 and res["f16_pressure_pct"] <= 1.0)
        res["cpu_seconds"] = round(time.time() - t0, 1)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main(sys.argv[1:] or ["128x128", "128x256", "256x256"])
