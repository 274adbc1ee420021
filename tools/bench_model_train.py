"""Training-loop throughput at the level of the reference's `Model` (opensplat.cpp:151-170: zero_grad, forward,
mainLoss, backward, optimizersStep, schedulersStep, afterTrain statistics) on one B200, config C2
(1M Gaussians, 1920x1080, SH degree 3):

  a) the reference's model.cpp, UNCHANGED, over the gsplat_b200 operators (libopensplat_model_b200.so): the three
     operators are ours, everything around them is the reference's ATen glue (cat, exp, normalize, sigmoid, 5 grouped
     conv2d for SSIM + autograd, six torch::optim::Adam, index_put statistics);
  b) the same C++ loop with gsb::modelForward / gsb::MainLoss (csrc/ops/fused_extras.hpp) opted in for the bodies
     of Model::forward / Model::mainLoss -- optimizers, schedulers and afterTrain still the reference's code;
  c) opensplat_b200.model.GaussianModel: same loop with all of that glue fused (SURVEY.md 8f rows 1-3).

    python tools/bench_model_train.py [--n 1000000] [--steps 30]"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def model_scene(n, W, H, seed=0):
    from opensplat_b200.scene import make_scene
    sc = make_scene(n, W, H, scale=0.02, sh_degree=3, opacity=(0.05, 0.6), seed=seed)
    f = np.float32
    # make_scene lays the Gaussians out for simple_trainer's w == 1 projection (x, y in [-1,1] ARE the NDC
    # coordinates).  Model::forward uses a true perspective P*V (ndc = (2 fx / W) x / z), so scale x, y by the view
    # depth to land every Gaussian on the same pixel with the same footprint (same M, same tile lists as C2).
    means = sc["means"].copy()
    z = means[:, 2] + 8.0
    means[:, 0] *= z * (W / (2.0 * sc["fx"]))
    means[:, 1] *= z * (H / (2.0 * sc["fy"]))
    p = {"means": means.astype(f), "scales": np.log(sc["scales"]).astype(f), "quats": sc["quats"],
         "featuresDc": np.ascontiguousarray(sc["coeffs"][:, 0, :]),
         "featuresRest": np.ascontiguousarray(sc["coeffs"][:, 1:, :]),
         "opacities": np.log(sc["opacities"] / (1 - sc["opacities"])).astype(f)}
    # Model::forward builds worldToCam = [D R0^T | -D R0^T T] with D = diag(1,-1,-1): this pose gives [I | (0,0,8)]
    c2w = np.array([[1, 0, 0, 0], [0, -1, 0, 0], [0, 0, -1, -8], [0, 0, 0, 1]], f)[None]
    return p, c2w, (sc["fx"], sc["fy"], sc["cx"], sc["cy"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--W", type=int, default=1920)
    ap.add_argument("--H", type=int, default=1080)
    a = ap.parse_args()
    dev = "cuda:0"
    from opensplat_b200 import cpp_ops
    from opensplat_b200.densify import RefineConfig
    from opensplat_b200.model import Camera, GaussianModel, PARAM_NAMES
    cpp_ops.ops()
    from oracle.build_model_b200 import OUT as MODEL_LIB
    torch.ops.load_library(MODEL_LIB)
    W, H = a.W, a.H
    p, c2w, (fx, fy, cx, cy) = model_scene(a.n, W, H)
    gts = torch.rand(1, H, W, 3)
    cfg = RefineConfig(warmup_length=10 ** 6)            # statistics every step, no refinement inside the timed loop
    out = {"workload": f"model_train_{a.n}_{W}x{H}_sh3", "steps": a.steps}
    probe = GaussianModel({k: torch.from_numpy(v) for k, v in p.items()}, cfg, device=dev)
    probe.forward(Camera(W, H, fx, fy, cx, cy, c2w[0]), 3001)
    out["visible"] = int((probe.radii > 0).sum())
    out["M"] = int(probe.numTilesHit.sum())
    del probe

    def run_cpp(first, steps, op=None):
        op = op or torch.ops.opensplat_b200_model.train
        params = [torch.from_numpy(p[x]).to(dev) for x in PARAM_NAMES]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = op(
            params, torch.from_numpy(c2w), gts, fx, fy, cx, cy, H, W, first, steps, 0.2, 1, 1000, 1, cfg.refine_every,
            cfg.warmup_length, cfg.reset_alpha_every, cfg.densify_grad_thresh, cfg.densify_size_thresh,
            cfg.stop_screen_size_at, cfg.split_screen_size, cfg.max_steps)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r
    run_cpp(3001, 3)                                     # warm-up (allocator, cudnn autotune of the SSIM convs)
    t_small, _ = run_cpp(3001, 2)
    t_big, r = run_cpp(3001, 2 + a.steps)
    dt = (t_big - t_small) / a.steps                     # subtract model construction + parameter upload
    out["reference_model_cpp_on_b200_ops"] = {"iters_per_s": 1.0 / dt, "ms_per_iter": dt * 1e3,
                                               "final_loss": float(r[0][-1])}

    # the same C++ loop with the opt-in one-liners of csrc/ops/fused_extras.hpp for the bodies of Model::forward /
    # Model::mainLoss (gsb::modelForward, gsb::MainLoss); optimizers, schedulers and afterTrain stay the reference's
    fused_op = torch.ops.opensplat_b200_model.train_fused
    run_cpp(3001, 3, fused_op)
    t_small, _ = run_cpp(3001, 2, fused_op)
    t_big, r = run_cpp(3001, 2 + a.steps, fused_op)
    dt = (t_big - t_small) / a.steps
    out["reference_loop_with_cpp_fused_opt_ins"] = {"iters_per_s": 1.0 / dt, "ms_per_iter": dt * 1e3,
                                                     "final_loss": float(r[0][-1])}

    model = GaussianModel({k: torch.from_numpy(v) for k, v in p.items()}, cfg, device=dev)
    cam = Camera(W, H, fx, fy, cx, cy, c2w[0])
    gt_pinned = gts[0].pin_memory()

    def step_py(step):
        model.optimizers_zero_grad()
        rgb = model.forward(cam, step)
        gt = gt_pinned.to(dev, non_blocking=True)        # the reference copies the ground truth H2D every step too
        loss = model.main_loss(rgb, gt, 0.2)
        loss.backward()
        model.optimizers_step()
        model.schedulers_step(step)
        model.after_train(step)
        return loss
    for s in range(3001, 3006):
        step_py(s)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(3006, 3006 + a.steps):
        loss = step_py(s)
    lv = float(loss.detach())
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / a.steps
    out["gaussian_model_fused_glue"] = {"iters_per_s": 1.0 / dt, "ms_per_iter": dt * 1e3, "final_loss": lv}
    out["speedup_fused_glue"] = out["gaussian_model_fused_glue"]["iters_per_s"] / out["reference_model_cpp_on_b200_ops"]["iters_per_s"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
