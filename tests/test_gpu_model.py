"""Drop-in check for the real caller of the hot path: the reference's model.cpp compiled UNCHANGED (-DUSE_CUDA)
against this repo's operator layer (oracle/build_model_b200.py -> libopensplat_model_b200.so) runs the body of the
reference training loop (opensplat.cpp:151-170: forward, mainLoss, backward, optimizersStep, schedulersStep,
afterTrain incl. two densifications) on the B200 back end.  What that run computes -- the reference's caller over THIS
repo's operators, so a regression baseline of this project rather than an output of the reference alone -- is stored
in tests/golden/b200_model_train.npz (tests/golden/make_golden_b200.py).  The host-side mirror
opensplat_b200.model.GaussianModel (fused activations / loss / Adam / topology edits) follows the same trajectory.

Both sides use the same CUDA kernels for the three operators; what differs is everything around them (ATen ops in
the reference's Model vs the fused kernels), so agreement is to round-off until the first refinement and, because a
refinement takes discrete decisions on values that differ in the last bits, to a looser bound afterwards."""
import os
import sys
import types

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from util import (PARAM_NAMES, TRAIN_REFINE, TRAIN_SEED, TRAIN_SH_INTERVAL, TRAIN_SSIM_WEIGHT,  # noqa: E402
                  TRAIN_STEPS, load_golden, make_problem)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference_run():
    """The reference's training loop on the B200 operators (golden): losses, counts, last image and the parameters
    at the stored rows."""
    g = load_golden("b200_model_train")
    ref_loss, ref_cnt = g["loss"], g["count"]
    assert np.isfinite(ref_loss).all() and ref_loss[18] < ref_loss[0]            # it trains
    assert ref_cnt[18] == len(make_problem()[0]["means"])
    assert ref_cnt[19] != ref_cnt[18] and ref_cnt[29] != ref_cnt[28]              # two refinements happened
    rows = torch.from_numpy(g["param_rows"]).to(DEV)
    return (ref_loss, ref_cnt, torch.from_numpy(g["rgb"]).to(DEV),
            {k: torch.from_numpy(g[k]).to(DEV) for k in PARAM_NAMES}, rows)


def _train_mirror():
    """The same loop (same problem, seed and schedule) over opensplat_b200.model.GaussianModel."""
    from opensplat_b200.densify import RefineConfig
    from opensplat_b200.model import Camera, GaussianModel
    p, c2w, gts, (fx, fy, cx, cy), H, W = make_problem()
    model = GaussianModel({k: torch.from_numpy(v) for k, v in p.items()}, RefineConfig(**TRAIN_REFINE),
                          sh_degree_interval=TRAIN_SH_INTERVAL, device=DEV)
    cams = [Camera(W, H, fx, fy, cx, cy, c2w[v]) for v in range(len(c2w))]
    gt_dev = torch.from_numpy(gts).to(DEV)
    torch.manual_seed(TRAIN_SEED)
    losses, counts, rgb = [], [], None
    for step in range(1, TRAIN_STEPS + 1):
        v = (step - 1) % len(cams)
        model.optimizers_zero_grad()
        rgb = model.forward(cams[v], step)
        loss = model.main_loss(rgb, gt_dev[v], TRAIN_SSIM_WEIGHT)
        loss.backward()
        losses.append(float(loss.detach()))
        model.optimizers_step()
        model.schedulers_step(step)
        model.after_train(step)
        counts.append(model.means.shape[0])
    return np.array(losses), np.array(counts), rgb.detach(), {k: getattr(model, k).detach() for k in PARAM_NAMES}


def _assert_follows(run, ref):
    (losses, counts, rgb, params), (ref_loss, ref_cnt, ref_rgb, ref_params, rows) = run, ref
    assert np.abs(losses[:20] - ref_loss[:20]).max() <= 5e-5, np.abs(losses[:20] - ref_loss[:20]).max()
    assert np.abs(counts - ref_cnt).max() <= 0.02 * ref_cnt.max(), (counts[[19, 29]], ref_cnt[[19, 29]])
    assert np.abs(losses - ref_loss).max() <= 5e-3, np.abs(losses - ref_loss).max()
    if np.array_equal(counts, ref_cnt):          # identical discrete decisions: the parameter sets line up row by row
        for k in PARAM_NAMES:
            a, b = params[k], ref_params[k]
            assert a.shape[0] == ref_cnt[-1] and a.shape[1:] == b.shape[1:], k
            a = a.index_select(0, rows)
            assert float((a - b).abs().max()) <= 2e-3 * (1.0 + float(b.abs().max())), k
        assert float((rgb - ref_rgb).abs().max()) <= 2e-2


def test_reference_model_cpp_unchanged_trains_on_b200_backend_and_mirror_follows():
    _assert_follows(_train_mirror(), _reference_run())


def _cpp_model_forward(model, cam, step):
    """What Model::forward becomes when a maintainer opts in (INTEGRATION.md; tests/native/model_driver.cpp's fused
    branch): gsb::modelForward on the down-scaled camera, xys / radii / image size kept for afterTrain."""
    sf = float(model.get_downscale_factor(step))
    h, w = int(float(cam.height) / sf), int(float(cam.width) / sf)
    rgb, xys, radii = torch.ops.opensplat_b200_test.model_forward(
        model.means, model.scales, model.quats, model.featuresDc, model.featuresRest, model.opacities,
        model.backgroundColor, cam.camToWorld, cam.fx / sf, cam.fy / sf, cam.cx / sf, cam.cy / sf, h, w,
        min(step // model.shDegreeInterval, model.shDegree))
    model.xys, model.radii, model.lastHeight, model.lastWidth = xys, radii, h, w
    return rgb


def test_cpp_model_forward_and_main_loss_opt_ins_follow_the_reference_training_loop(monkeypatch):
    """SURVEY 8f row 1 from C++: gsb::modelForward (host-side camera matrices, tile bounds, background early return,
    then ProjectGaussiansActivated -> SphericalHarmonicsRgb -> RasterizeGaussiansClamped) and gsb::MainLoss
    (csrc/ops/fused_extras.hpp) as the forward and loss of the mirror's training loop (its Adam, schedule and
    afterTrain) follow the reference's UNCHANGED model.cpp loop on the same operators (golden): same losses to
    rounding, same refinement decisions."""
    from opensplat_b200 import cpp_ops, model as model_mod
    from opensplat_b200.model import Camera, GaussianModel
    o = cpp_ops.ops()
    torch.ops.load_library(os.path.join(ROOT, "tests", "native", "_build", "libopensplat_b200_test_ops.so"))

    # no Gaussian in view (camera turned away from the scene): the background, as Model::forward returns it
    p, c2w, _, (fx, fy, cx, cy), H, W = make_problem()
    away = c2w[len(c2w) // 2].copy()
    away[:3, :3] = away[:3, :3] @ np.diag([-1.0, 1.0, -1.0]).astype(np.float32)
    m = GaussianModel({k: torch.from_numpy(v) for k, v in p.items()}, device=DEV)
    cam = Camera(W, H, fx, fy, cx, cy, away)
    m.backgroundColor = torch.tensor([0.25, 0.5, 0.75], device=DEV)
    rgb = _cpp_model_forward(m, cam, 1)
    assert int(m.radii.sum()) == 0 and rgb.shape == (m.lastHeight, m.lastWidth, 3)
    assert torch.equal(rgb, m.backgroundColor.repeat(m.lastHeight, m.lastWidth, 1))

    monkeypatch.setattr(GaussianModel, "forward", _cpp_model_forward)
    monkeypatch.setattr(model_mod.ops, "MainLoss", types.SimpleNamespace(apply=o.main_loss))
    _assert_follows(_train_mirror(), _reference_run())


def test_gaussian_model_save_matches_reference_writer(tmp_path):
    """GaussianModel.save == Model::save bytes (golden from the reference's own writer)."""
    from opensplat_b200.model import GaussianModel
    from util import load_golden, scene_edit_inputs
    g = load_golden("scene_edit_save")
    p = scene_edit_inputs(int(g["n"]), int(g["k"]), int(g["seed"]))[0]
    model = GaussianModel({k: torch.from_numpy(v) for k, v in p.items()}, device=DEV)
    fn = str(tmp_path / "out.ply")
    model.save(fn, step=int(g["step"]))
    assert open(fn, "rb").read() == g["ply"].tobytes()
