"""Generate the run.py fixtures from the REAL reference implementation.

Needs a checkout of facebookresearch/VideoPose3D (CPU only):

    python tests/golden/make_run_py_golden.py --reference /path/to/VideoPose3D

1. `run_py_epoch_1.bin`: the checkpoint the unmodified reference `run.py` writes after one epoch on
   the synthetic dataset of tools/make_synthetic_h36m.py (the arguments of
   tests/test_run_py_smoke.py): `model_pos` of a TemporalModel arc 3,3, C = 32, the amsgrad Adam
   state, lr, epoch and the generator's random state, in run.py's own format (run.py:600-608).
2. `run_py_resume.json`: training resumed from that checkpoint the way run.py's loop drives it
   (root joint zeroed, mpjpe, backward, Adam step; run.py:401-420) with the reference's
   TemporalModelOptimized1f, its `mpjpe` and torch.optim.Adam on seeded batches, then the
   reference's TemporalModel in eval mode on the trained weights: the per-step losses and the
   final predictions.  tests/test_gpu_run_py.py repeats this with this package's classes.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import temporal_model_oracle as orc  # noqa: E402

RUN_ARGS = ["-k", "gt", "-arc", "3,3", "-ch", "32", "-e", "1", "-b", "128", "-str", "S1", "-ste", "S9",
            "--checkpoint-frequency", "1"]
# resumed training: batch shapes and seeds (tests/test_gpu_run_py.py draws the same batches)
RESUME = dict(arc=[3, 3], channels=32, batch=256, steps=12, eval_batch=16, eval_frames=15,
              input_seed=300, target_seed=400, eval_seed=500)


def batches(cfg):
    """The seeded (2-D input, 3-D target) batches of the resumed training and the eval input."""
    t = 1
    for w in cfg["arc"]:
        t *= w
    out = []
    for i in range(cfg["steps"]):
        x = orc.make_input(cfg["batch"], t, 17, 2, seed=cfg["input_seed"] + i)
        g = torch.Generator().manual_seed(cfg["target_seed"] + i)
        y = torch.randn(cfg["batch"], 1, 17, 3, generator=g) * 0.3
        y[:, :, 0] = 0                                   # run.py:407
        out.append((x, y))
    x_eval = orc.make_input(cfg["eval_batch"], cfg["eval_frames"], 17, 2, seed=cfg["eval_seed"])
    return out, x_eval


def resume_reference(checkpoint, cfg, dtype=torch.float32):
    from common.loss import mpjpe
    from common.model import TemporalModel, TemporalModelOptimized1f
    chk = torch.load(checkpoint, map_location="cpu", weights_only=False)
    train = TemporalModelOptimized1f(17, 2, 17, filter_widths=cfg["arc"], dropout=0.0,
                                     channels=cfg["channels"])
    train.load_state_dict(chk["model_pos"])
    train = train.to(dtype).train()
    opt = torch.optim.Adam(train.parameters(), lr=chk["lr"], amsgrad=True)
    opt.load_state_dict(chk["optimizer"])
    data, x_eval = batches(cfg)
    losses = []
    for x, y in data:
        opt.zero_grad()
        loss = mpjpe(train(x.to(dtype)), y.to(dtype))
        loss.backward()
        opt.step()
        losses.append(loss.item())
    ev = TemporalModel(17, 2, 17, filter_widths=cfg["arc"], channels=cfg["channels"])
    ev.load_state_dict(train.state_dict())
    ev = ev.to(dtype).eval()
    with torch.no_grad():
        pred = ev(x_eval.to(dtype))
    return losses, pred.double()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True, help="checkout of facebookresearch/VideoPose3D")
    args = ap.parse_args()
    ref = os.path.abspath(args.reference)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="4")
    work = tempfile.mkdtemp()
    try:
        subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "make_synthetic_h36m.py"),
                               "--reference", ref, "--out", os.path.join(work, "data"), "--frames", "80",
                               "--subjects", "S1,S9", "--actions", "Walking"], cwd=work, env=env)
        subprocess.check_call([sys.executable, os.path.join(ref, "run.py")] + RUN_ARGS + ["-c", "ckpt"],
                              cwd=work, env=env)
        checkpoint = os.path.join(HERE, "run_py_epoch_1.bin")
        shutil.copy(os.path.join(work, "ckpt", "epoch_1.bin"), checkpoint)
    finally:
        shutil.rmtree(work, ignore_errors=True)

    sys.path.insert(0, ref)
    losses, pred = resume_reference(checkpoint, RESUME)
    losses64, pred64 = resume_reference(checkpoint, RESUME, torch.float64)
    print("float32 vs float64 reference: max rel loss diff",
          max(abs(a - b) / abs(b) for a, b in zip(losses, losses64)),
          "prediction rel err", float((pred - pred64).abs().max() / pred64.abs().max()))
    with open(os.path.join(HERE, "run_py_resume.json"), "w") as f:
        json.dump({"config": RESUME, "torch": torch.__version__, "losses": losses,
                   "pred_shape": list(pred.shape), "pred": pred.flatten().tolist()}, f)
        f.write("\n")
    print("losses", losses)


if __name__ == "__main__":
    main()
