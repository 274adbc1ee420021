import os
import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name + ".npz")))


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def image_close(a, b, tol=1e-5, flip=4.5e-3, frac=1e-3):
    """SURVEY 8c tolerance statement: >= (1-frac) of pixels within tol, the rest (isolated
    alpha-threshold flips) bounded by 1/255 (+ slack)."""
    d = np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max(axis=-1)
    bad = d > tol
    return bad.mean() <= frac and d.max() <= flip, (float(bad.mean()), float(d.max()))


# ---- scene-edit (densification / export) inputs, regenerated from a seed on both sides of every comparison ----
PARAM_NAMES = ("means", "scales", "quats", "featuresDc", "featuresRest", "opacities")


def scene_edit_inputs(n, sh_bases, seed, max_dim=640):
    """Random Gaussian set + Adam moments + per-step (v_xy, radii) draws whose statistics straddle every
    threshold Model::afterTrain compares against (model.cpp:343-349,375,439-451).  numpy PCG64: stable across
    versions, so fixtures only need to store the reference's OUTPUTS."""
    rng = np.random.default_rng(seed)
    f = np.float32
    p = {
        "means": rng.uniform(-1, 1, (n, 3)).astype(f),
        # exp(scales) log-uniform in [0.002, 1.2]: below / above densifySizeThresh 0.01 and cullScaleThresh 0.5 (also /1.6)
        "scales": np.log(np.exp(rng.uniform(np.log(0.002), np.log(1.2), (n, 3)))).astype(f),
        "quats": (rng.standard_normal((n, 4)) * rng.uniform(0.5, 2.0, (n, 1))).astype(f),
        "featuresDc": rng.uniform(-2.5, 2.5, (n, 3)).astype(f),
        "featuresRest": (rng.standard_normal((n, sh_bases - 1, 3)) * 0.2).astype(f),
        "opacities": rng.uniform(-4.0, 2.0, (n, 1)).astype(f),       # sigmoid in [0.018, 0.88]: around 0.1
    }
    m = {k: (rng.standard_normal(v.shape) * 1e-3).astype(f) for k, v in p.items()}
    v = {k: (rng.uniform(0, 1, v_.shape) * 1e-6).astype(f) for k, v_ in p.items()}
    steps = []
    for _ in range(3):
        radii = rng.integers(-20, 130, n).astype(np.int32)           # radii / 640 around 0.05 and 0.15; many <= 0
        v_xy = (rng.standard_normal((n, 2)) * rng.uniform(0, 2.5e-6, (n, 1))).astype(f)   # avg norm * 320 around 2e-4
        v_xy[radii <= 0] = 0
        steps.append((v_xy, radii))
    return p, m, v, steps


# ---- the short training run of tests/test_gpu_model.py (tests/golden/make_golden_b200.py records the reference's) ----
TRAIN_STEPS, TRAIN_SEED, TRAIN_SSIM_WEIGHT, TRAIN_SH_INTERVAL = 34, 11, 0.2, 8
TRAIN_REFINE = dict(num_cameras=3, refine_every=10, warmup_length=15, reset_alpha_every=30, densify_grad_thresh=2e-5,
                    densify_size_thresh=0.05, stop_screen_size_at=4000, split_screen_size=0.05, max_steps=200)


def make_problem(n=4000, V=3, H=96, W=128, k=4, seed=5):
    rng = np.random.default_rng(seed)
    f = np.float32
    p = {
        "means": (rng.uniform(-1, 1, (n, 3)) * np.array([1.6, 1.2, 0.5])).astype(f),
        "scales": np.log(rng.uniform(0.02, 0.12, (n, 3))).astype(f),
        "quats": rng.standard_normal((n, 4)).astype(f),
        "featuresDc": rng.uniform(-1.5, 1.5, (n, 3)).astype(f),
        "featuresRest": (rng.standard_normal((n, k - 1, 3)) * 0.1).astype(f),
        "opacities": rng.uniform(-2.0, 1.0, (n, 1)).astype(f),
    }
    c2w = np.tile(np.eye(4, dtype=f), (V, 1, 1))
    for v in range(V):                       # OpenGL-style poses on a circle of radius 4, looking at the origin
        a = 0.25 * (v - (V - 1) / 2)
        c2w[v, :3, :3] = np.array([[np.cos(a), 0, -np.sin(a)], [0, 1, 0], [np.sin(a), 0, np.cos(a)]], dtype=f)
        c2w[v, :3, 3] = np.array([-4.0 * np.sin(a), 0.0, 4.0 * np.cos(a)], dtype=f)
    yy, xx = np.mgrid[0:H, 0:W]
    gts = np.stack([np.stack([0.5 + 0.5 * np.sin(0.07 * xx + v), 0.5 + 0.5 * np.cos(0.05 * yy - v),
                              0.5 + 0.25 * np.sin(0.03 * (xx + yy))], -1) for v in range(V)]).astype(f)
    return p, c2w, gts, (0.9 * W, 0.9 * W, W / 2.0, H / 2.0), H, W
