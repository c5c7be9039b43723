"""CPU -- SURVEY §8 row f3.

The full protocol needs a checkout of the reference (skipped without one):
  1. tools/make_synthetic_h36m.py writes a dataset pair the UNMODIFIED reference run.py accepts:
     one training epoch + evaluation with the reference's own model runs to completion;
  2. the checkpoint it saves loads into this package's classes: `model_pos` into TemporalModel
     (strict) and `optimizer` into FusedAdam -- the checkpoint round trip of run.py:600-608;
  3. tools/run_reference.py runs the same unchanged script with the model classes swapped in: on a
     machine without CUDA that must end in this package's "no CPU fallback" error, raised from
     inside run.py's training loop (i.e. the script really constructed and called our classes).
Step 2 also runs everywhere on the checkpoint such a run wrote, stored as
tests/golden/run_py_epoch_1.bin (tests/golden/make_run_py_golden.py).
"""
import os
import subprocess
import sys

import pytest
import torch

import videopose3d_b200 as vp
from videopose3d_b200.optim import FusedAdam

from oracle import stage_ref

REFERENCE = stage_ref.reference_dir() or "/root/reference"   # staged archive on the GPU box
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GOLDEN_CHECKPOINT = os.path.join(ROOT, "tests", "golden", "run_py_epoch_1.bin")

RUN_ARGS = ["-k", "gt", "-arc", "3,3", "-ch", "32", "-e", "1", "-b", "128", "-str", "S1", "-ste", "S9",
            "--checkpoint-frequency", "1"]


def _run(cmd, cwd):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="4")
    return subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True, timeout=600)


def _check_checkpoint_loads_into_our_classes(path):
    chk = torch.load(path, map_location="cpu", weights_only=False)
    ours = vp.TemporalModel(17, 2, 17, filter_widths=[3, 3], channels=32)
    ours.load_state_dict(chk["model_pos"])                # strict: identical keys and shapes
    ours_1f = vp.TemporalModelOptimized1f(17, 2, 17, filter_widths=[3, 3], channels=32)
    ours_1f.load_state_dict(chk["model_pos"])             # the two classes share checkpoints
    opt = FusedAdam(ours_1f.parameters(), lr=1e-3, amsgrad=True)
    opt.load_state_dict(chk["optimizer"])
    assert abs(opt.param_groups[0]["lr"] - chk["lr"]) < 1e-12
    for p in ours_1f.parameters():
        assert set(opt.state[p]) >= {"step", "exp_avg", "exp_avg_sq", "max_exp_avg_sq"}
        assert opt.state[p]["exp_avg"].shape == p.shape


def test_reference_run_py_checkpoint_loads_into_our_classes():
    _check_checkpoint_loads_into_our_classes(GOLDEN_CHECKPOINT)


@pytest.mark.skipif(not os.path.exists(os.path.join(REFERENCE, "run.py")),
                    reason="reference checkout not present")
def test_unmodified_run_py_trains_on_synthetic_data_and_checkpoints_interchange(tmp_path):
    work = str(tmp_path)
    r = _run([sys.executable, os.path.join(ROOT, "tools", "make_synthetic_h36m.py"), "--reference",
              REFERENCE, "--out", os.path.join(work, "data"), "--frames", "80", "--subjects", "S1,S9",
              "--actions", "Walking"], work)
    assert r.returncode == 0, r.stderr[-2000:]
    r = _run([sys.executable, os.path.join(REFERENCE, "run.py")] + RUN_ARGS + ["-c", "ckpt"], work)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "Protocol #1" in r.stdout                      # the final evaluation ran
    _check_checkpoint_loads_into_our_classes(os.path.join(work, "ckpt", "epoch_1.bin"))

    if not torch.cuda.is_available():
        r = _run([sys.executable, os.path.join(ROOT, "tools", "run_reference.py"), "--reference",
                  REFERENCE, "--swap", "model,loss,optim", "--"] + RUN_ARGS + ["-c", "ckpt2"], work)
        assert r.returncode != 0
        assert "no CPU fallback" in r.stderr and "run.py" in r.stderr
