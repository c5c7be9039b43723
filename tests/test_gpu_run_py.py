"""GPU: the reference's run.py, UNCHANGED, on the B200 with this package's classes swapped in
(SURVEY §8 row f3; reference call sites run.py:21, 171-184, 311-420, 652-721).

The reference reaches the GPU box only as the archive staged by oracle/stage_ref.py; the test is
skipped where neither /root/reference nor the archive exists.  Protocol:
  1. tools/make_synthetic_h36m.py writes a Human3.6M-format dataset pair;
  2. the reference's own classes train epoch 1 and save a checkpoint (common starting point:
     run.py never seeds torch, so two cold starts would differ by their initialisation);
  3. epoch 2 is run twice from that checkpoint (`--resume`, same optimizer state and generator
     stream): with the reference's classes on PyTorch/cuDNN (TF32 off) and with model / loss /
     optimizer swapped for videopose3d_b200 (training kernels in their fp32-faithful mode).  The
     epoch-2 training loss, eval-mode losses and the final Protocol #1-#3 / velocity errors must
     agree;
  4. the same with the device-resident generators swapped in as well and the default (bf16)
     training kernels: same numbers within bf16 noise;
  5. checkpoint round trip: the epoch-2 checkpoint written by OUR classes is evaluated by the
     reference's classes (`--evaluate`) and vice versa.

Without the reference, test_resume_from_run_py_checkpoint_trains_like_the_reference checks step 3
against stored reference results (tests/golden/make_run_py_golden.py): training resumed from a
checkpoint the unchanged run.py wrote, driven as run.py's loop drives it, must reproduce the
reference's per-step losses and its eval-mode predictions on the trained weights.
"""
import json
import os
import re
import shutil
import subprocess
import sys

import pytest
import torch

from oracle import stage_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

ARGS = ["-k", "gt", "-arc", "3,3,3", "-ch", "64", "-b", "256", "-drop", "0", "-str", "S1,S5",
        "-ste", "S9", "--checkpoint-frequency", "1", "-lrd", "1.0"]
EPOCH_RE = re.compile(r"^\[(\d+)\] time \S+ lr \S+ 3d_train (\S+) 3d_eval (\S+) 3d_valid (\S+)", re.M)
FINAL_RE = {k: re.compile(p + r" ([0-9.eE+-]+) mm") for k, p in {
    "p1": r"Protocol #1 Error \(MPJPE\):", "p2": r"Protocol #2 Error \(P-MPJPE\):",
    "p3": r"Protocol #3 Error \(N-MPJPE\):", "vel": r"Velocity Error \(MPJVE\):"}.items()}


def _run(cmd, cwd, **env):
    e = dict(os.environ, NVIDIA_TF32_OVERRIDE="0", TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD="1",
             OMP_NUM_THREADS="4", CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0"))
    e.update(env)
    r = subprocess.run(cmd, cwd=cwd, env=e, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, (cmd, r.stdout[-1500:], r.stderr[-3000:])
    return r.stdout


def _epoch(out, epoch):
    rows = {int(m.group(1)): tuple(float(g) for g in m.groups()[1:]) for m in EPOCH_RE.finditer(out)}
    assert epoch in rows, out[-2000:]
    return rows[epoch]


def _final(out):
    got = {}
    for k, rx in FINAL_RE.items():
        vals = [float(v) for v in rx.findall(out)]
        assert vals, (k, out[-2000:])
        got[k] = sum(vals) / len(vals)       # mean over the per-action blocks evaluate() prints
    return got


def _close(a, b, rel):
    return abs(a - b) <= rel * max(abs(a), abs(b), 1e-12)


def _tol(key, base):
    # the velocity error differentiates the prediction over time: a few-1e-4 perturbation of the
    # poses (fp16 inference) moves it by ~0.5 % while Protocols #1-#3 move by 1e-5
    return 4 * base if key == "vel" else base


def test_run_py_unchanged_trains_and_evaluates_like_the_reference(tmp_path):
    ref = stage_ref.reference_dir()
    if ref is None:
        pytest.skip("no reference checkout and no staged archive (oracle/stage_ref.py)")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    work = str(tmp_path)
    py = sys.executable
    launcher = [py, os.path.join(ROOT, "tools", "run_reference.py"), "--reference", ref]
    _run([py, os.path.join(ROOT, "tools", "make_synthetic_h36m.py"), "--reference", ref, "--out",
          os.path.join(work, "data"), "--frames", "300", "--subjects", "S1,S5,S9", "--actions",
          "Walking,Directions 1"], work)
    # epoch 1 with the reference's own classes -> common checkpoint
    _run([py, os.path.join(ref, "run.py")] + ARGS + ["-e", "1", "-c", "ck_ref"], work)
    for d in ("ck_ours", "ck_fast"):
        os.makedirs(os.path.join(work, d))
        shutil.copy(os.path.join(work, "ck_ref", "epoch_1.bin"), os.path.join(work, d, "epoch_1.bin"))
    resume = ["-e", "2", "-r", "epoch_1.bin"]
    out_ref = _run([py, os.path.join(ref, "run.py")] + ARGS + resume + ["-c", "ck_ref"], work)
    out_ours = _run(launcher + ["--swap", "model,loss,optim", "--"] + ARGS + resume + ["-c", "ck_ours"],
                    work, VP3D_TRAIN_PRECISION="bf16x3", VP3D_PRECISION="bf16x3")
    out_fast = _run(launcher + ["--swap", "model,loss,optim,generators", "--"] + ARGS + resume +
                    ["-c", "ck_fast"], work)
    e_ref, e_ours, e_fast = _epoch(out_ref, 2), _epoch(out_ours, 2), _epoch(out_fast, 2)
    f_ref, f_ours, f_fast = _final(out_ref), _final(out_ours), _final(out_fast)
    print("epoch 2 (3d_train, 3d_eval, 3d_valid): reference", e_ref, "ours fp32-faithful", e_ours,
          "ours default + device generators", e_fast)
    print("final: reference", f_ref, "ours", f_ours, "ours fast", f_fast)
    for a, b in zip(e_ref, e_ours):
        assert _close(a, b, 5e-3), (e_ref, e_ours)
    for k in f_ref:
        assert _close(f_ref[k], f_ours[k], 5e-3), (k, f_ref, f_ours)
    # default kernels (bf16 training, fp16 inference) + device-resident generators
    for a, b in zip(e_ref, e_fast):
        assert _close(a, b, 3e-2), (e_ref, e_fast)
    for k in f_ref:
        assert _close(f_ref[k], f_fast[k], _tol(k, 3e-2)), (k, f_ref, f_fast)
    # checkpoint round trip in both directions (run.py:600-608 writes, :204-210 reads)
    # (run.py:216-219 loads `model_traj` whenever the key exists, and its own supervised
    # checkpoints carry the key with value None -- a quirk of the reference: drop the key, which
    # is how the published checkpoints look)
    for src, dst in (("ck_ours/epoch_2.bin", "ck_ref/ours_2.bin"), ("ck_ref/epoch_2.bin", "ck_ours/ref_2.bin")):
        chk = torch.load(os.path.join(work, src), map_location="cpu", weights_only=False)
        chk.pop("model_traj", None)
        torch.save(chk, os.path.join(work, dst))
    ev_ref_on_ours = _final(_run([py, os.path.join(ref, "run.py")] + ARGS +
                                 ["--evaluate", "ours_2.bin", "-c", "ck_ref"], work))
    ev_ours_on_ref = _final(_run(launcher + ["--swap", "model", "--"] + ARGS +
                                 ["--evaluate", "ref_2.bin", "-c", "ck_ours"], work))
    print("reference classes on our checkpoint", ev_ref_on_ours, "our classes (fp16 eval) on the "
          "reference checkpoint", ev_ours_on_ref)
    for k in f_ref:
        assert _close(ev_ref_on_ours[k], f_ours[k], 5e-3), (k, ev_ref_on_ours, f_ours)
        assert _close(ev_ours_on_ref[k], f_ref[k], _tol(k, 5e-3)), (k, ev_ours_on_ref, f_ref)


def test_resume_from_run_py_checkpoint_trains_like_the_reference(cuda_device):
    import numpy as np
    import videopose3d_b200 as vp
    from videopose3d_b200 import loss as vloss
    from videopose3d_b200.optim import FusedAdam

    golden = os.path.join(ROOT, "tests", "golden")
    sys.path.insert(0, golden)
    try:
        import make_run_py_golden as mk
    finally:
        sys.path.remove(golden)
    with open(os.path.join(golden, "run_py_resume.json")) as f:
        ref = json.load(f)
    cfg = ref["config"]
    chk = torch.load(os.path.join(golden, "run_py_epoch_1.bin"), map_location="cpu", weights_only=False)
    # the fp32-faithful training / inference kernels, as in the run.py comparison above
    train = vp.TemporalModelOptimized1f(17, 2, 17, filter_widths=cfg["arc"], dropout=0.0,
                                        channels=cfg["channels"])
    train.load_state_dict(chk["model_pos"])
    train = train.to(cuda_device).train().set_train_precision("bf16x3")
    opt = FusedAdam(train.parameters(), lr=chk["lr"], amsgrad=True)
    opt.load_state_dict(chk["optimizer"])
    data, x_eval = mk.batches(cfg)
    losses = []
    for x, y in data:
        opt.zero_grad()
        loss = vloss.mpjpe(train(x.to(cuda_device)), y.to(cuda_device))
        loss.backward()
        opt.step()
        losses.append(loss.item())
    ev = vp.TemporalModel(17, 2, 17, filter_widths=cfg["arc"], channels=cfg["channels"])
    ev.load_state_dict({k: v.cpu() for k, v in train.state_dict().items()})
    ev = ev.to(cuda_device).eval().set_precision("bf16x3")
    with torch.no_grad():
        pred = ev(x_eval.to(cuda_device)).double().cpu().numpy()
    want = np.array(ref["pred"]).reshape(ref["pred_shape"])
    print("losses: reference", ref["losses"], "ours", losses)
    for a, b in zip(ref["losses"], losses):
        assert _close(a, b, 5e-3), (ref["losses"], losses)
    assert pred.shape == want.shape
    err = float(np.abs(pred - want).max() / np.abs(want).max())
    print(f"eval prediction after {len(losses)} steps: rel err {err:.2e}")
    assert err <= 5e-3
