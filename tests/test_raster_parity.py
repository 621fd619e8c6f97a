"""GPU parity: our rasterizer (through the C ABI / drop-in Python API) against the
reference's own CUDA code on identical seeded inputs (its outputs are stored in
tests/golden/parity_test_raster_parity.npz, see tests/ref_golden.py).

Bars (BASELINE.json north_star): bit-exact radii, tile keys, sorted order, tile ranges;
colour and depth within 1e-4 max-abs; gradients within 1e-3 relative (of the tensor's
max-abs, since the reference's own float atomics are run-to-run nondeterministic)."""
import numpy as np
import pytest
import torch

from b200gs import synthetic as syn
from ref_golden import Golden

pytestmark = pytest.mark.gpu

COLOR_TOL = 1e-4
GRAD_RTOL = 1e-3


def _ours_forward(cam, bg, act, sh_degree=3, colors_precomp=None, cov3D_precomp=None, requires_grad=False):
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    st = GaussianRasterizationSettings(cam.image_height, cam.image_width, cam.tanfovx, cam.tanfovy, bg, 1.0,
                                       cam.viewmatrix, cam.projmatrix, sh_degree, cam.campos, False, False)
    ras = GaussianRasterizer(st)
    inp = {k: v.clone().requires_grad_(requires_grad) for k, v in act.items()}
    means2D = torch.zeros_like(inp["means3D"], requires_grad=requires_grad)
    kw = dict(means3D=inp["means3D"], means2D=means2D, opacities=inp["opacities"])
    if colors_precomp is not None:
        cp = colors_precomp.clone().requires_grad_(requires_grad); kw["colors_precomp"] = cp; inp["colors_precomp"] = cp
    else:
        kw["shs"] = inp["shs"]
    if cov3D_precomp is not None:
        c3 = cov3D_precomp.clone().requires_grad_(requires_grad); kw["cov3D_precomp"] = c3; inp["cov3D_precomp"] = c3
    else:
        kw["scales"] = inp["scales"]; kw["rotations"] = inp["rotations"]
    color, radii, depth = ras(**kw)
    return color, radii, depth, inp, means2D


def _export(P, R, cam, fn_out):
    from b200gs.rasterizer import _C
    geom, binb, img = fn_out
    H, W = cam.image_height, cam.image_width
    def get(name, dt):
        return _C.export_state(name, P, R, W, H, geom, binb, img).cpu().numpy().view(dt)
    return get


def _scene(P, W, H, mu, device="cuda"):
    raw = syn.make_gaussians(P, scale_mu=mu, device=device)
    act = syn.activated(raw)
    cam = syn.make_camera(W, H, device=device)
    return act, cam


# BASELINE.json's full sizes: C3 (1M, 1280x720), C4 (1920x1080), C5 (5M at 3840x2160)
_FULL = [(1000000, 1280, 720, 0.010), (1000000, 1920, 1080, 0.004), (5000000, 3840, 2160, 0.004)]


@pytest.mark.parametrize("P,W,H,mu", [(2000, 64, 48, 0.02), (20000, 200, 120, 0.01), (200000, 512, 512, 0.004),
                                      (200000, 512, 512, 0.010)] + _FULL)
def test_forward_bit_exact_and_image(P, W, H, mu, request):
    from b200gs.rasterizer import _C
    ref = Golden(request)
    act, cam = _scene(P, W, H, mu)
    bg = torch.tensor([0.1, 0.2, 0.3], device="cuda")
    out = _C.rasterize_gaussians(bg, act["means3D"], torch.Tensor([]), act["opacities"], act["scales"],
                                 act["rotations"], 1.0, torch.Tensor([]), cam.viewmatrix, cam.projmatrix,
                                 cam.tanfovx, cam.tanfovy, H, W, act["shs"], 3, cam.campos, False, False)
    R, color, depth, radii, geom, binb, img = out
    torch.cuda.synchronize()
    assert R == ref.value("R")
    assert ref.equal("radii", radii)
    get = _export(P, R, cam, (geom, binb, img))
    vis = radii.cpu().numpy() > 0
    assert ref.equal("tiles_touched", get("tiles_touched", np.uint32))
    assert ref.equal("keys", get("keys", np.uint64))
    assert ref.equal("point_list", get("point_list", np.uint32))
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    assert ref.equal("ranges", get("ranges", np.uint32)[: 2 * tiles])
    # per-Gaussian projected state (visible ones; the reference leaves culled slots stale)
    assert ref.equal("depths", get("depths", np.float32)[vis])
    assert ref.equal("means2D", get("means2D", np.float32).reshape(-1, 2)[vis])
    assert ref.equal("cov3D", get("cov3D", np.float32).reshape(-1, 6)[vis])
    assert ref.equal("conic_opacity", get("conic_opacity", np.float32).reshape(-1, 4)[vis])
    assert ref.maxdiff("rgb", get("rgb", np.float32).reshape(-1, 3)[vis]) <= 2e-6
    assert ref.equal("n_contrib", get("n_contrib", np.uint32))
    assert ref.maxdiff("accum_alpha", get("accum_alpha", np.float32)) <= 1e-6
    assert ref.maxdiff("color", color) <= COLOR_TOL
    assert ref.maxdiff("depth", depth) <= COLOR_TOL


@pytest.mark.parametrize("P,W,H,mu,depth_grad", [(20000, 200, 120, 0.01, True), (200000, 512, 512, 0.004, False),
                                                 (200000, 512, 512, 0.010, True)] + [c + (True,) for c in _FULL])
def test_backward_gradients(P, W, H, mu, depth_grad, request):
    ref = Golden(request)
    act, cam = _scene(P, W, H, mu)
    bg = torch.tensor([0.0, 0.0, 0.0], device="cuda")
    g = torch.Generator(device="cpu").manual_seed(7)
    gt = torch.rand(3, H, W, generator=g).cuda()
    color, radii, depth, inp, means2D = _ours_forward(cam, bg, act, requires_grad=True)
    loss = (color - gt).abs().mean()
    wd = torch.randn(1, H, W, generator=g).cuda() / (H * W) if depth_grad else None
    if depth_grad:
        loss = loss + (depth * wd).sum()
    loss.backward()
    # the reference's backward was given OUR colour's sign pattern, so both sides saw the same upstream gradient
    pairs = [("means3D", inp["means3D"].grad), ("means2D", means2D.grad), ("sh", inp["shs"].grad),
             ("opacity", inp["opacities"].grad), ("scales", inp["scales"].grad), ("rotations", inp["rotations"].grad)]
    for name, ours in pairs:
        assert ours is not None, name
        r = ref.rel(name, ours)
        assert r <= GRAD_RTOL, f"{name}: rel err {r:.3e}"


def test_precomputed_colors_and_cov(request):
    ref = Golden(request)
    P, W, H = 20000, 160, 96
    act, cam = _scene(P, W, H, 0.01)
    bg = torch.tensor([0.3, 0.1, 0.0], device="cuda")
    g = torch.Generator().manual_seed(3)
    colors = torch.rand(P, 3, generator=g).cuda()
    # covariance the way scene/gaussian_model.py:31-35 builds it: (R S)(R S)^T, upper triangle
    q = act["rotations"]; s = act["scales"]
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    Rm = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                      2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                      2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1).reshape(-1, 3, 3)
    L = Rm * s[:, None, :]
    Sig = L @ L.transpose(1, 2)
    cov = torch.stack([Sig[:, 0, 0], Sig[:, 0, 1], Sig[:, 0, 2], Sig[:, 1, 1], Sig[:, 1, 2], Sig[:, 2, 2]], -1).contiguous()
    color, radii, depth, inp, means2D = _ours_forward(cam, bg, act, colors_precomp=colors, cov3D_precomp=cov,
                                                      requires_grad=True)
    assert ref.equal("radii", radii)
    assert ref.maxdiff("color", color) <= COLOR_TOL
    gt = torch.rand(3, H, W, generator=g).cuda()
    (color - gt).pow(2).mean().backward()
    # the reference's backward was given dL = 2 (OUR colour - gt) / (3 H W)
    assert ref.rel("colors", inp["colors_precomp"].grad) <= GRAD_RTOL
    assert ref.rel("cov3D", inp["cov3D_precomp"].grad) <= GRAD_RTOL
    assert ref.rel("means3D", inp["means3D"].grad) <= GRAD_RTOL
    assert ref.rel("opacity", inp["opacities"].grad) <= GRAD_RTOL


def test_edge_cases_empty_and_behind_camera():
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    cam = syn.make_camera(40, 24, device="cuda")
    bg = torch.tensor([0.5, 0.25, 0.75], device="cuda")
    st = GaussianRasterizationSettings(24, 40, cam.tanfovx, cam.tanfovy, bg, 1.0, cam.viewmatrix, cam.projmatrix, 3,
                                       cam.campos, False, False)
    ras = GaussianRasterizer(st)
    # P = 0: background image, no error (rasterize_points.cu:82 guards P != 0)
    z = lambda *s: torch.zeros(*s, device="cuda")
    color, radii, depth = ras(means3D=z(0, 3), means2D=z(0, 3), opacities=z(0, 1), shs=z(0, 16, 3), scales=z(0, 3),
                              rotations=z(0, 4))
    assert radii.numel() == 0 and color.shape == (3, 24, 40)
    # all Gaussians behind the camera: radii 0, pure background
    raw = syn.make_gaussians(500, device="cuda"); act = syn.activated(raw)
    act["means3D"] = act["means3D"] + torch.tensor([0, 0, -20.0], device="cuda")
    color, radii, depth = ras(means3D=act["means3D"], means2D=z(500, 3), opacities=act["opacities"], shs=act["shs"],
                              scales=act["scales"], rotations=act["rotations"])
    assert int((radii > 0).sum()) == 0
    assert torch.allclose(color, bg[:, None, None].expand_as(color))
    assert float(depth.abs().max()) == 0.0
    # argument validation mirrors RAST/diff_gaussian_rasterization/__init__.py:192-196
    with pytest.raises(Exception):
        ras(means3D=act["means3D"], means2D=z(500, 3), opacities=act["opacities"])
    with pytest.raises(Exception):
        ras(means3D=act["means3D"], means2D=z(500, 3), opacities=act["opacities"], shs=act["shs"], scales=act["scales"])
    vis = ras.markVisible(act["means3D"])
    assert vis.dtype == torch.bool and int(vis.sum()) == 0


def test_empty_model_renders_the_background_through_the_whole_path():
    """Zero Gaussians (everything pruned) through engine.render: deformation field, activations, rasterizer, to8b."""
    from b200gs import engine, output, synthetic as syn
    dev = torch.device("cuda", 0)
    raw = syn.make_gaussians(0, device=dev)
    m = engine.GaussianState(raw).to(dev)
    cam = syn.make_camera(64, 48, device=dev)
    bg = torch.tensor([0.25, 0.5, 0.75], device=dev)
    for stage in ("coarse", "fine"):
        with torch.no_grad():
            pkg = engine.render(cam, m, bg, stage=stage)
        assert pkg["render"].shape == (3, 48, 64) and pkg["radii"].numel() == 0
        assert torch.equal(pkg["render"], bg[:, None, None].expand(3, 48, 64))
        assert float(pkg["depth"].abs().max()) == 0.0
    q = output.to8b(pkg["render"])
    assert q.shape == (48, 64, 3) and q[0, 0].tolist() == [63, 127, 191]
