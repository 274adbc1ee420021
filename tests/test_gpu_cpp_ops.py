"""GPU: the C++/libtorch operator layer (the actual drop-in: same class names / signatures as the
reference's project_gaussians.hpp, rasterize_gaussians.hpp, spherical_harmonics.hpp) and the reference's
UNCHANGED simple_trainer.cpp compiled against it (the losses it printed, stored as golden data)."""
import numpy as np
import pytest
import torch

from opensplat_b200 import cpp_ops, ops
from util import load_golden, rel_l2, image_close

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.parametrize("name,gtol", [("chain_tight_100x72", 2e-3), ("chain_bg_quat_128x96", 2e-3)])
def test_cpp_operator_chain_vs_reference_golden(name, gtol):
    g = load_golden(name)
    o = cpp_ops.ops()
    fx, fy, cx, cy = [float(v) for v in g["intrins"]]
    H, W = [int(v) for v in g["hw"]]
    means, scales, quats = (cu(g[k]).requires_grad_() for k in ("means", "scales", "quats"))
    colors, opac = cu(g["colors"]).requires_grad_(), cu(g["opacities"]).requires_grad_()
    xys, depths, radii, conics, nth, cov3d = o.project_gaussians(means, scales, 1.0, quats, cu(g["viewmat"]),
                                                                 cu(g["projmat"]), fx, fy, cx, cy, H, W, 0.01)
    xys.retain_grad()
    img = o.rasterize_gaussians(xys, depths, radii, conics, nth, colors, opac, H, W, cu(g["background"]))
    ok, stats = image_close(img.detach().cpu().numpy(), g["ref_img"], tol=5e-5)
    assert ok, stats
    (img * cu(g["wgt"])).sum().backward()
    for got, ref in [(xys.grad, "ref_v_xy"), (colors.grad, "ref_v_colors"), (opac.grad, "ref_v_opacity"),
                     (means.grad, "ref_v_means"), (scales.grad, "ref_v_scales"), (quats.grad, "ref_v_quats")]:
        assert rel_l2(got.cpu().numpy(), g[ref]) <= gtol
    # the python mirror drives the same C ABI -> bit-identical
    m2, s2, q2 = (cu(g[k]).requires_grad_() for k in ("means", "scales", "quats"))
    c2, o2 = cu(g["colors"]).requires_grad_(), cu(g["opacities"]).requires_grad_()
    p = ops.ProjectGaussians.apply(m2, s2, 1.0, q2, cu(g["viewmat"]), cu(g["projmat"]), fx, fy, cx, cy, H, W,
                                   ops.tile_bounds(W, H))
    img2 = ops.RasterizeGaussians.apply(p[0], p[1], p[2], p[3], p[4], c2, o2, H, W, cu(g["background"]))
    (img2 * cu(g["wgt"])).sum().backward()
    assert torch.equal(img, img2) and torch.equal(means.grad, m2.grad) and torch.equal(quats.grad, q2.grad)


def test_cpp_sh_and_bin_and_sort():
    o = cpp_ops.ops()
    g = load_golden("sh_deg3")
    co = cu(g["coeffs"]).requires_grad_()
    col = o.spherical_harmonics(3, cu(g["viewdirs"]), co)
    (col * cu(g["wgt"])).sum().backward()
    assert np.abs(col.detach().cpu().numpy() - g["ref_colors_d3"]).max() <= 2e-5
    assert np.abs(co.grad.cpu().numpy() - g["ref_v_coeffs_d3"]).max() <= 2e-6
    gg = load_golden("chain_tight_100x72")
    fx, fy, cx, cy = [float(v) for v in gg["intrins"]]
    H, W = [int(v) for v in gg["hw"]]
    xys, depths, radii, conics, nth, _ = o.project_gaussians(cu(gg["means"]), cu(gg["scales"]), 1.0, cu(gg["quats"]),
                                                             cu(gg["viewmat"]), cu(gg["projmat"]), fx, fy, cx, cy, H, W,
                                                             0.01)
    cum = torch.cumsum(nth, 0, dtype=torch.int32)
    tb = ops.tile_bounds(W, H)
    isect, gids, ks, gs, bins = o.bin_and_sort_gaussians(xys.shape[0], int(cum[-1]), xys, depths, radii, cum, tb[0], tb[1])
    ref = torch.sort(isect, stable=True)
    assert torch.equal(ks, ref.values) and torch.equal(gs, gids[ref.indices])


def _python_simple_trainer(width, height, n, iters, lr=0.01):
    """simple_trainer.cpp:84-203 restated with the python mirror operators (same seeds, same math)."""
    torch.manual_seed(0)
    gt = torch.ones(height, width, 3)
    gt[: height // 2, : width // 2, :] = torch.tensor([1.0, 0.0, 0.0])
    gt[height // 2:, width // 2:, :] = torch.tensor([0.0, 0.0, 1.0])
    gt = gt.to(DEV)
    focal = 0.5 * width / np.tan(0.5 * np.pi / 2.0)
    means = 2.0 * (torch.rand(n, 3) - 0.5)
    scales = torch.rand(n, 3)
    rgbs = torch.rand(n, 3)
    u, v, w = torch.rand(n, 1), torch.rand(n, 1), torch.rand(n, 1)
    means, scales, rgbs, u, v, w = (t.to(DEV) for t in (means, scales, rgbs, u, v, w))
    quats = torch.cat([torch.sqrt(1 - u) * torch.sin(2 * np.pi * v), torch.sqrt(1 - u) * torch.cos(2 * np.pi * v),
                       torch.sqrt(u) * torch.sin(2 * np.pi * w), torch.sqrt(u) * torch.cos(2 * np.pi * w)], -1)
    opac = torch.ones(n, 1, device=DEV)
    view = torch.eye(4, device=DEV)
    view[2, 3] = 8.0
    bg = torch.zeros(3, device=DEV)
    for t in (means, scales, quats, rgbs, opac):
        t.requires_grad_()
    opt = torch.optim.Adam([rgbs, means, scales, opac, quats], lr, foreach=False)
    tb = ops.tile_bounds(width, height)
    losses = []
    for _ in range(iters):
        p = ops.ProjectGaussians.apply(means, scales, 1, quats, view, view, focal, focal, width // 2, height // 2,
                                       height, width, tb)
        img = ops.RasterizeGaussians.apply(p[0], p[1], p[2], p[3], p[4], torch.sigmoid(rgbs), torch.sigmoid(opac),
                                           height, width, bg)
        loss = torch.nn.functional.mse_loss(img, gt)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses


def test_reference_simple_trainer_losses_on_b200_backend_followed_by_mirror():
    """The losses the reference's UNCHANGED simple_trainer.cpp printed when compiled against this repo's operator layer
    (oracle/build_simple_trainer.py; stored by tests/golden/make_golden_b200.py as a regression baseline of these
    operators under the reference's caller) are followed by its restatement over the python mirror operators."""
    g = load_golden("b200_simple_trainer")
    iters, n, W, H = (int(g[k]) for k in ("iters", "points", "width", "height"))
    losses = list(g["losses"])
    assert len(losses) == iters
    assert losses[-1] < 0.8 * losses[0]                      # it trains
    py = _python_simple_trainer(W, H, n, iters)
    assert abs(py[0] - losses[0]) <= 1e-5 * max(1.0, abs(py[0]))   # same forward on the same seeded scene
    assert np.abs(np.array(py) - np.array(losses)).max() <= 2e-3 * max(py)  # same trajectory


# ---- optional fused replacements for the ATen glue in Model (csrc/ops/fused_extras.hpp) ----------------------
def test_cpp_main_loss_vs_reference_golden():
    o = cpp_ops.ops()
    g = load_golden("loss_45x70")
    dev = "cuda:0"
    rend = torch.from_numpy(g["rendered"]).to(dev).requires_grad_()
    loss = o.main_loss(rend, torch.from_numpy(g["gt"]).to(dev), float(g["ssim_weight"]))
    (2.0 * loss).backward()
    assert abs(float(loss.detach()) - float(g["ref_loss"])) <= 2e-6                  # vs the reference's Model::mainLoss
    assert rel_l2(rend.grad.cpu().numpy(), 2.0 * g["ref_v_rendered"]) <= 2e-5
    r2 = torch.from_numpy(g["rendered"]).to(dev).requires_grad_()
    l2 = ops.MainLoss.apply(r2, torch.from_numpy(g["gt"]).to(dev), float(g["ssim_weight"]))
    l2.backward()
    # same kernels behind both layers; the scalar is an atomic float sum (last-bit order dependence)
    assert abs(float(l2.detach()) - float(loss.detach())) <= 1e-7
    assert float((2.0 * r2.grad - rend.grad).abs().max()) <= 1e-9


def test_cpp_adam_step_matches_torch_adam():
    o = cpp_ops.ops()
    torch.manual_seed(3)
    p = torch.randn(100_003, device="cuda:0")
    q = p.clone().requires_grad_()
    opt = torch.optim.Adam([q], lr=0.005)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    for step in range(1, 5):
        g = torch.randn_like(p) * 0.1
        q.grad = g.clone()
        opt.step()
        o.adam_step_(p, g, m, v, 0.005, step, 0.9, 0.999, 1e-8)
        assert float((p - q.detach()).abs().max()) <= 2e-6
    st = opt.state[q]
    assert float((m - st["exp_avg"]).abs().max()) <= 1e-7 and float((v - st["exp_avg_sq"]).abs().max()) <= 1e-8


def test_cpp_densify_stats_matches_python_path():
    from opensplat_b200.densify import Densifier
    o = cpp_ops.ops()
    dev = "cuda:0"
    torch.manual_seed(4)
    n, H, W = 50_000, 300, 480
    dn = Densifier()
    gn, vc, ms = (torch.empty(n, device=dev) for _ in range(3))
    for i in range(3):
        v_xy = torch.randn(n, 2, device=dev) * 1e-4
        radii = torch.randint(-5, 60, (n,), device=dev, dtype=torch.int32)
        dn.accumulate(v_xy, radii, H, W)
        o.densify_stats_(v_xy, radii, H, W, i == 0, gn, vc, ms)
    assert torch.equal(gn, dn.xys_grad_norm) and torch.equal(vc, dn.vis_counts) and torch.equal(ms, dn.max_2d_size)


def test_cpp_fused_activation_and_colour_operators_match_python_mirrors():
    """gsb::ActivateGaussians / gsb::SphericalHarmonicsRgb (csrc/ops/fused_extras.hpp: the opt-in one-liners for
    model.cpp:148-150,176-177,186-192,200) against the Python autograd mirrors over the same C ABI -- forward and
    gradients bit-identical (same kernels), and against the unfused op sequence to rounding."""
    co = cpp_ops.ops()
    torch.manual_seed(3)
    n, K = 4099, 16
    means = torch.randn(n, 3, device=DEV)
    cam = torch.tensor([0.2, 0.1, -7.5])                      # host tensor: the operator moves it
    ls, rq, ol = (torch.randn(n, k, device=DEV).requires_grad_() for k in (3, 4, 1))
    dc = torch.randn(n, 3, device=DEV).requires_grad_()
    rest = (0.3 * torch.randn(n, K - 1, 3, device=DEV)).requires_grad_()
    w = [torch.randn(n, k, device=DEV) for k in (3, 4, 1, 3)]

    def run(act, shrgb):
        for t in (ls, rq, ol, dc, rest):
            t.grad = None
        s, q, o, vd = act(means, ls, rq, ol, cam)
        rgbs = shrgb(2, means, cam, dc, rest)
        ((s * w[0]).sum() + (q * w[1]).sum() + (o * w[2]).sum() + (rgbs * w[3]).sum()).backward()
        return [t.detach().clone() for t in (s, q, o, vd, rgbs)] + [t.grad.clone() for t in (ls, rq, ol, dc, rest)]

    a = run(co.activate_gaussians, co.spherical_harmonics_rgb)
    b = run(ops.ActivateGaussians.apply, ops.SphericalHarmonicsRgb.apply)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    # unfused reference sequence
    vd = (means - cam.to(DEV)) / (means - cam.to(DEV)).norm(dim=-1, keepdim=True)
    ref = torch.clamp_min(co.spherical_harmonics(2, vd, torch.cat([dc[:, None, :], rest], 1).detach()) + 0.5, 0.0)
    assert float((a[4] - ref).abs().max()) <= 3e-6
    assert float((a[0] - torch.exp(ls.detach())).abs().max()) <= 2e-6 * float(torch.exp(ls.detach()).max())


def _raw_model_scene(n, W, H, seed):
    """A make_scene scene expressed in the model's RAW parameters (log-scales, un-normalised quaternions, opacity
    logits) plus bright colours, so that the activations and the clamp all have something to do."""
    from opensplat_b200.scene import make_scene
    sc = make_scene(n, W, H, scale=0.25, sh_degree=0, opacity=(0.05, 0.9), seed=seed)
    rng = np.random.default_rng(seed)
    raw = {
        "means": torch.from_numpy(sc["means"]).to(DEV),
        "ls": torch.from_numpy(np.log(sc["scales"])).to(DEV),
        "rq": torch.from_numpy(sc["quats"] * rng.uniform(0.5, 2.0, (n, 1)).astype(np.float32)).to(DEV),
        "ol": torch.from_numpy(np.log(sc["opacities"] / (1 - sc["opacities"])).astype(np.float32)).reshape(n, 1).to(DEV),
        "colors": torch.from_numpy(rng.uniform(0.0, 1.6, (n, 3)).astype(np.float32)).to(DEV),
    }
    cam = dict(view=torch.from_numpy(sc["viewmat"]).to(DEV), proj=torch.from_numpy(sc["projmat"]).to(DEV),
               fx=sc["fx"], fy=sc["fy"], cx=sc["cx"], cy=sc["cy"])
    return raw, cam


@pytest.mark.parametrize("n,W,H", [(20_000, 320, 208), (1, 33, 17)])
def test_fused_projection_and_clamped_rasterizer_match_the_unfused_sequence(n, W, H):
    """SURVEY 8f row 1, the last glue ops of Model::forward: exp / normalize / sigmoid folded into the projection
    (ProjectGaussiansActivated) and clamp_max(rgb, 1) folded into the blend kernels (RasterizeGaussiansClamped),
    against the sequence model.cpp:148-150,152-165,200,213-222 runs -- torch activations + ProjectGaussians +
    RasterizeGaussians + torch.clamp_max -- with torch autograd through it.  The clamped rasterizer has the same
    arithmetic as the plain one, so image and gradients must be BIT-identical; the projection differs by rounding
    only (one quaternion normalisation instead of two, expf inside the no-FMA translation unit)."""
    raw, cam = _raw_model_scene(n, W, H, seed=n + 5)
    tb = ops.tile_bounds(W, H)
    bg = torch.tensor([1.0, 0.4, 0.9], device=DEV)
    w_img = torch.randn(H, W, 3, device=DEV)
    leaves = [raw[k].clone().requires_grad_() for k in ("means", "ls", "rq", "ol", "colors")]

    def unfused(means, ls, rq, ol, colors):
        scales, quats, opac = torch.exp(ls), rq / rq.norm(dim=-1, keepdim=True), torch.sigmoid(ol)
        xys, depths, radii, conics, nth, _ = ops.ProjectGaussians.apply(
            means, scales, 1.0, quats, cam["view"], cam["proj"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], H, W, tb)
        rgb = ops.RasterizeGaussians.apply(xys, depths, radii, conics, nth, colors, opac, H, W, bg)
        return torch.clamp_max(rgb, 1.0), (xys, depths, radii, conics, nth, opac), rgb

    def fused(means, ls, rq, ol, colors):
        xys, depths, radii, conics, nth, _, opac = ops.ProjectGaussiansActivated.apply(
            means, ls, 1.0, rq, ol, cam["view"], cam["proj"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], H, W, tb)
        rgb = ops.RasterizeGaussiansClamped.apply(xys, depths, radii, conics, nth, colors, opac, H, W, bg)
        return rgb, (xys, depths, radii, conics, nth, opac), None

    def grads(fn):
        for t in leaves:
            t.grad = None
        img, proj_out, raw_img = fn(*leaves)
        (img * w_img).sum().backward()
        return img.detach(), proj_out, [t.grad.clone() for t in leaves], raw_img

    img_u, pu, gu, raw_img = grads(unfused)
    img_f, pf, gf, _ = grads(fused)
    # --- projection: same integers (a radius could flip by rounding; none may in more than 0.1 % of the Gaussians)
    same = (pu[2] == pf[2]) & (pu[4] == pf[4])
    assert float(same.float().mean()) >= 0.999
    for a, b, tol in ((pu[0], pf[0], 0.0), (pu[1], pf[1], 0.0), (pu[3], pf[3], 1e-4), (pu[5], pf[5], 1e-6)):   # xys, depths: means only
        d = (a - b).abs()[same] if a.shape[0] == same.shape[0] else (a - b).abs()
        assert float(d.max()) <= tol * max(1.0, float(b.abs().max())), float(d.max())
    # --- the clamp really cut something, image within rounding of the unfused one, gradients too
    if n > 1:
        assert float((raw_img > 1.0).float().mean()) > 0.02
    assert float(img_f.max()) <= 1.0
    assert float((img_u - img_f).abs().max()) <= 2e-4
    for a, b in zip(gu, gf):
        assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) <= 2e-3, rel_l2(a.cpu().numpy(), b.cpu().numpy())

    # --- the clamped rasterizer alone, on identical inputs: bit-identical image and gradients
    xys, depths, radii, conics, nth, opac = [t.detach() for t in pf]
    outs = []
    for op, clamp_after in ((ops.RasterizeGaussians, True), (ops.RasterizeGaussiansClamped, False)):
        xl, cl, col, ol_ = (t.clone().requires_grad_() for t in (xys, conics, raw["colors"], opac))
        img = op.apply(xl, depths, radii, cl, nth, col, ol_, H, W, bg)
        if clamp_after:
            img = torch.clamp_max(img, 1.0)
        (img * w_img).sum().backward()
        outs.append([img.detach(), xl.grad, cl.grad, col.grad, ol_.grad])
    for a, b in zip(*outs):
        assert torch.equal(a, b)

    # --- C++ twins (gsb::ProjectGaussiansActivated / gsb::RasterizeGaussiansClamped): same kernels, same bits
    co = cpp_ops.ops()

    def fused_cpp(means, ls, rq, ol, colors):
        xys, depths, radii, conics, nth, _, opac = co.project_gaussians_activated(
            means, ls, 1.0, rq, ol, cam["view"], cam["proj"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], H, W, 0.01)
        rgb = co.rasterize_gaussians_clamped(xys, depths, radii, conics, nth, colors, opac, H, W, bg)
        return rgb, (xys, depths, radii, conics, nth, opac), None

    img_c, pc, gc, _ = grads(fused_cpp)
    assert torch.equal(img_c, img_f)
    for a, b in zip(pc, pf):
        assert torch.equal(a, b)
    for a, b in zip(gc, gf):
        assert torch.equal(a, b)


def test_clamped_rasterizer_on_the_generic_fallback_path():
    """Tile lists longer than the in-shared-memory sort takes (the operator falls back to the generic global sort and
    gsb_pack_records): the clamp flag must travel down that branch as well."""
    from opensplat_b200.scene import make_scene
    n, W, H = 24_000, 64, 48
    sc = make_scene(n, W, H, scale=0.5, sh_degree=0, opacity=(0.0045, 0.01), seed=n)
    sc["means"][:, 0] = 0.25 + sc["means"][:, 0] * 0.05
    sc["means"][:, 1] = sc["means"][:, 1] * 0.05
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    tb = ops.tile_bounds(W, H)
    _, xys, depths, radii, conics, nth = ops.project_gaussians_forward(
        t(sc["means"]), t(sc["scales"]), 1.0, t(sc["quats"]), t(sc["viewmat"]), t(sc["projmat"]), sc["fx"], sc["fy"],
        sc["cx"], sc["cy"], H, W, tb)
    colors = torch.from_numpy(np.random.default_rng(2).uniform(0.5, 3.0, (n, 3)).astype(np.float32)).to(DEV)
    opac, bg = t(sc["opacities"]), torch.tensor([0.2, 0.9, 0.5], device=DEV)
    w_img = torch.randn(H, W, 3, device=DEV)
    outs = []
    for op, clamp_after in ((ops.RasterizeGaussians, True), (ops.RasterizeGaussiansClamped, False)):
        col, ol_ = colors.clone().requires_grad_(), opac.clone().requires_grad_()
        img = op.apply(xys, depths, radii, conics, nth, col, ol_, H, W, bg)
        if clamp_after:
            raw_img = img.detach()
            img = torch.clamp_max(img, 1.0)
        (img * w_img).sum().backward()
        outs.append([img.detach(), col.grad, ol_.grad])
    assert float((raw_img > 1.0).float().mean()) > 0.001
    for a, b in zip(*outs):
        assert torch.equal(a, b)
