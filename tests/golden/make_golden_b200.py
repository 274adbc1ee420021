"""Generates the golden vectors of the two drop-in checks on the GPU: what the reference's UNCHANGED
simple_trainer.cpp and model.cpp (-DUSE_CUDA) compute when compiled against this repo's operator layer
(oracle/build_simple_trainer.py, oracle/build_model_b200.py -> oracle/_ref; built by __graft_entry__.build() where the
reference tree exists).  They run THIS project's operators under the reference's callers, so the files are a
regression baseline of this project, not independent reference data.  Needs a CUDA device:

    python tests/golden/make_golden_b200.py [OUT_DIR]        # default: tests/golden

  b200_simple_trainer.npz : the losses simple_trainer_b200 prints (tests/test_gpu_cpp_ops.py)
  b200_model_train.npz    : losses, Gaussian counts, last image and parameters of the reference's training loop on
                            the problem of tests/util.py make_problem (tests/test_gpu_model.py); the parameters at
                            PARAM_ROWS seeded rows (param_rows), which keeps the file below 1 MB"""
import os
import re
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from util import (PARAM_NAMES, TRAIN_REFINE, TRAIN_SEED, TRAIN_SH_INTERVAL, TRAIN_SSIM_WEIGHT,  # noqa: E402
                  TRAIN_STEPS, make_problem)

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
SIMPLE_TRAINER = dict(width=256, height=256, points=2000, iters=30)
PARAM_ROWS = 1024


def simple_trainer(out):
    a = SIMPLE_TRAINER
    r = subprocess.run([os.path.join(REF_DIR, "simple_trainer_b200"), "--width", str(a["width"]), "--height",
                        str(a["height"]), "--points", str(a["points"]), "--iters", str(a["iters"])],
                       capture_output=True, text=True, timeout=300, check=True)
    assert "Using CUDA" in r.stdout, r.stdout[-2000:]
    losses = np.array([float(x) for x in re.findall(r"Loss: ([0-9.eE+-]+)", r.stdout)], np.float64)
    assert len(losses) == a["iters"], r.stdout[-2000:]
    np.savez_compressed(os.path.join(out, "b200_simple_trainer.npz"), losses=losses,
                        **{k: np.int64(v) for k, v in a.items()})


def model_train(out):
    from opensplat_b200 import cpp_ops
    cpp_ops.ops()                            # libopensplat_b200_ops.so, which the model library links against
    torch.ops.load_library(os.path.join(REF_DIR, "libopensplat_model_b200.so"))
    p, c2w, gts, (fx, fy, cx, cy), H, W = make_problem()
    c = TRAIN_REFINE
    params = [torch.from_numpy(p[x]).cuda() for x in PARAM_NAMES]
    r = torch.ops.opensplat_b200_model.train(
        params, torch.from_numpy(c2w), torch.from_numpy(gts), fx, fy, cx, cy, H, W, 1, TRAIN_STEPS, TRAIN_SSIM_WEIGHT,
        TRAIN_SEED, TRAIN_SH_INTERVAL, c["num_cameras"], c["refine_every"], c["warmup_length"],
        c["reset_alpha_every"], c["densify_grad_thresh"], c["densify_size_thresh"], c["stop_screen_size_at"],
        c["split_screen_size"], c["max_steps"])
    torch.cuda.synchronize()
    n = r[3].shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, PARAM_ROWS), replace=False))
    arrays = {"loss": r[0].numpy(), "count": r[1].numpy(), "rgb": r[2].cpu().numpy(), "param_rows": rows}
    arrays.update({k: t.cpu().numpy()[rows] for k, t in zip(PARAM_NAMES, r[3:9])})
    np.savez_compressed(os.path.join(out, "b200_model_train.npz"), **arrays)


if __name__ == "__main__":
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.abspath(__file__))
    os.makedirs(out, exist_ok=True)
    simple_trainer(out)
    model_train(out)
    for f in sorted(os.listdir(out)):
        print(f, os.path.getsize(os.path.join(out, f)))
