"""LBM_FORCE_EVERY and LBM_FORCE_BOXES are checked before the GPU is touched: each bad value ends in
die() with a message that names it (a bad box by its index), and no output file is written.
These paths end before lbm_gpu_create, so they run on CPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "d2q9-bgk")
PARAMS = os.path.join(ROOT, "inputs", "input_128x128.params")
OBST = os.path.join(ROOT, "inputs", "obstacles_128x128.dat")

pytestmark = pytest.mark.skipif(not os.path.exists(EXE) or not os.path.exists(PARAMS),
                                reason="host binary or shipped inputs not built (make)")


def refused(tmp_path, env):
    e = dict(os.environ)
    for k in ("LBM_FORCE_EVERY", "LBM_FORCE_BOXES", "LBM_CHECKPOINT", "LBM_CHECKPOINT_EVERY", "LBM_RESTART"):
        e.pop(k, None)
    e.update(env)
    r = subprocess.run([EXE, PARAMS, OBST], cwd=str(tmp_path), env=e, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 1, (r.returncode, r.stderr)
    assert r.stderr.startswith("Error at line "), r.stderr
    assert os.listdir(str(tmp_path)) == []
    return r.stderr


@pytest.mark.parametrize("k", ["0", "-4", "ten", "", "5x", "99999999999"])
def test_force_every_must_be_a_positive_step_count(tmp_path, k):
    assert "LBM_FORCE_EVERY must be a positive number of steps" in refused(tmp_path, {"LBM_FORCE_EVERY": k})


def test_boxes_need_force_every(tmp_path):
    assert "LBM_FORCE_BOXES needs LBM_FORCE_EVERY" in refused(tmp_path, {"LBM_FORCE_BOXES": "0,0,10,10"})


@pytest.mark.parametrize("spec,index,why", [
    ("1,2,3", 0, "is not four integers"),
    ("0,0,10,10;1,2,3,4,5", 1, "is not four integers"),
    ("0,0,10,10;;0,0,1,1", 1, "is not four integers"),
    ("0,0,10,10;", 1, "is not four integers"),
    ("a,0,10,10", 0, "is not four integers"),
    ("0,0,129,10", 0, "is not within"),
    ("0,0,128,129", 0, "is not within"),
    ("5,0,4,10", 0, "is not within"),
    ("0,0,10,10;0,7,10,6", 1, "is not within"),
    ("-1,0,10,10", 0, "is not within"),
])
def test_a_bad_box_is_named(tmp_path, spec, index, why):
    msg = refused(tmp_path, {"LBM_FORCE_EVERY": "10", "LBM_FORCE_BOXES": spec})
    assert ("LBM_FORCE_BOXES: box %d " % index) in msg and why in msg, msg


def test_too_many_boxes(tmp_path):
    msg = refused(tmp_path, {"LBM_FORCE_EVERY": "10", "LBM_FORCE_BOXES": ";".join(["0,0,1,1"] * 257)})
    assert "more than 256 boxes" in msg
