"""GPU parity of the rasterizer configurations the reference can reach but the headline tests do not: active SH degree 0 / 1 / 2
(train_4DGS.py:153 raises it every 1000 iterations, `oneupSHdegree`), `scale_modifier != 1`, a non-zero background in the
BACKWARD (backward.cu:531-536: the `bg . dL_dpixel` term of dL_dalpha), `colors_precomp` with a depth gradient, the
`prefiltered` flag, and `markVisible` against the reference's own `checkFrustum` (rasterizer_impl.cu:54-66, :141-153) on a
scene that straddles the near plane z = 0.2.

Everything is compared with the reference's own CUDA code (its outputs on these inputs are stored in
tests/golden/parity_test_raster_parity_configs.npz, see tests/ref_golden.py).  Two gradient metrics:
  * max-abs error relative to the tensor's max-abs  <= 1e-3   (what tests/test_raster_parity.py uses);
  * PER-ELEMENT relative error |ours - ref| / |ref| over the stored sample elements with |ref| >= 1e-2 max|ref|  <= 1e-3.
    (With the reference at hand the bound was max(1e-3, 8 x the reference's own run-to-run noise in the same metric): it
    accumulates with float atomics, so two runs of ITS backward differ.  The stored values carry no such noise.)
"""
import numpy as np
import pytest
import torch

from b200gs import synthetic as syn
from ref_golden import Golden

pytestmark = pytest.mark.gpu

COLOR_TOL = 1e-4
GRAD_RTOL = 1e-3
FLOOR = 1e-2


def _rel_elementwise(ref, name, ours, floor=FLOOR):
    """max over the sampled {i : |ref_i| >= floor * max|ref|} of |ours_i - ref_i| / |ref_i| (0 if the set is empty)."""
    a, b = ref.sampled(name, ours)
    m = np.abs(b) >= floor * ref.maxabs(name, ours)
    if not m.any():
        return 0.0
    return float((np.abs(a[m] - b[m]) / np.abs(b[m])).max())


def _settings(cam, bg, sh_degree, scale_modifier=1.0, prefiltered=False):
    from diff_gaussian_rasterization import GaussianRasterizationSettings
    return GaussianRasterizationSettings(cam.image_height, cam.image_width, cam.tanfovx, cam.tanfovy, bg, scale_modifier,
                                         cam.viewmatrix, cam.projmatrix, sh_degree, cam.campos, prefiltered, False)


def _check_grads(ref, pairs):
    worst = {}
    for name, ours in pairs:
        assert ours is not None, name
        r = ref.rel(name, ours)
        assert r <= GRAD_RTOL, f"{name}: max-abs relative error {r:.3e}"
        e = _rel_elementwise(ref, name, ours)
        assert e <= GRAD_RTOL, f"{name}: per-element relative error {e:.3e}"
        worst[name] = (r, e)
    return worst


@pytest.mark.parametrize("D,scale_modifier,bgv", [(0, 1.0, (0.0, 0.0, 0.0)), (1, 1.0, (0.3, 0.6, 0.1)), (2, 0.7, (1.0, 1.0, 1.0)),
                                                   (3, 0.7, (0.2, 0.5, 0.9)), (3, 1.3, (0.0, 0.0, 0.0))])
def test_sh_degree_scale_modifier_background(D, scale_modifier, bgv, request):
    from diff_gaussian_rasterization import GaussianRasterizer
    ref = Golden(request)
    P, W, H = 60000, 320, 208
    raw = syn.make_gaussians(P, scale_mu=0.012, seed=100 + D, device="cuda")
    act = syn.activated(raw)
    with torch.no_grad():          # enough energy in the higher bands for their gradients to be visible
        act["shs"][:, 1:] *= 6.0
    cam = syn.orbit_cameras(3, W, H, device="cuda")[1]
    bg = torch.tensor(bgv, device="cuda")
    inp = {k: v.clone().requires_grad_(True) for k, v in act.items()}
    means2D = torch.zeros_like(inp["means3D"], requires_grad=True)
    color, radii, depth = GaussianRasterizer(_settings(cam, bg, D, scale_modifier))(
        means3D=inp["means3D"], means2D=means2D, opacities=inp["opacities"], shs=inp["shs"], scales=inp["scales"],
        rotations=inp["rotations"])
    assert ref.equal("radii", radii)
    assert ref.maxdiff("color", color) <= COLOR_TOL
    assert ref.maxdiff("depth", depth) <= COLOR_TOL
    g = torch.Generator().manual_seed(11 + D)
    dL_dcolor = (torch.randn(3, H, W, generator=g) / (3 * H * W)).cuda()
    dL_ddepth = (torch.randn(1, H, W, generator=g) / (H * W)).cuda()
    torch.autograd.backward([color, depth], [dL_dcolor, dL_ddepth])
    pairs = [("means3D", inp["means3D"].grad), ("means2D", means2D.grad), ("sh", inp["shs"].grad),
             ("opacity", inp["opacities"].grad), ("scales", inp["scales"].grad), ("rotations", inp["rotations"].grad)]
    worst = _check_grads(ref, pairs)
    # coefficients above the active degree get exactly zero gradient, like the reference (backward.cu:47-137)
    n_active = (D + 1) ** 2
    assert float(inp["shs"].grad[:, n_active:].abs().max()) == 0.0 if n_active < 16 else True
    print({k: tuple(f"{x:.1e}" for x in v) for k, v in worst.items()})


def test_colors_precomp_with_depth_gradient_and_background(request):
    from diff_gaussian_rasterization import GaussianRasterizer
    ref = Golden(request)
    P, W, H = 50000, 256, 160
    raw = syn.make_gaussians(P, scale_mu=0.012, seed=31, device="cuda")
    act = syn.activated(raw)
    cam = syn.orbit_cameras(4, W, H, device="cuda")[2]
    bg = torch.tensor([0.7, 0.2, 0.4], device="cuda")
    g = torch.Generator().manual_seed(3)
    colors = torch.rand(P, 3, generator=g).cuda()
    inp = {k: act[k].clone().requires_grad_(True) for k in ("means3D", "opacities", "scales", "rotations")}
    cp = colors.clone().requires_grad_(True)
    means2D = torch.zeros_like(inp["means3D"], requires_grad=True)
    color, radii, depth = GaussianRasterizer(_settings(cam, bg, 3, 0.9))(
        means3D=inp["means3D"], means2D=means2D, opacities=inp["opacities"], colors_precomp=cp, scales=inp["scales"],
        rotations=inp["rotations"])
    assert ref.equal("radii", radii)
    assert ref.maxdiff("color", color) <= COLOR_TOL and ref.maxdiff("depth", depth) <= COLOR_TOL
    dL_dcolor = (torch.randn(3, H, W, generator=g) / (3 * H * W)).cuda()
    dL_ddepth = (torch.randn(1, H, W, generator=g) / (H * W)).cuda()
    torch.autograd.backward([color, depth], [dL_dcolor, dL_ddepth])
    _check_grads(ref, [("colors", cp.grad), ("means3D", inp["means3D"].grad), ("means2D", means2D.grad),
                       ("opacity", inp["opacities"].grad), ("scales", inp["scales"].grad), ("rotations", inp["rotations"].grad)])


def _straddling_scene(P, device="cuda"):
    """Gaussians spread along the optical axis from well behind the camera to far in front of it, with a dense band around
    the near plane (view-space z = 0.2, auxiliary.h:154), including a slab of points within a few ULPs of it."""
    g = torch.Generator().manual_seed(77)
    cam = syn.make_camera(96, 64, device=device)           # camera at z = -4.5 looking down +z: view z = world z + 4.5
    xyz = torch.rand(P, 3, generator=g) * 2.0 - 1.0
    z_view = torch.cat([torch.rand(P // 2, generator=g) * 12.0 - 4.0,                    # [-4, 8]
                        0.2 + (torch.rand(P // 4, generator=g) - 0.5) * 1e-2,            # +- 5e-3 around the plane
                        0.2 + (torch.randint(-4, 5, (P - P // 2 - P // 4,), generator=g).float() * 2.0 ** -22)])  # a few ULPs
    xyz[:, 2] = z_view - 4.5
    return cam, xyz.to(device).contiguous()


def test_mark_visible_matches_reference_check_frustum(request):
    from diff_gaussian_rasterization import GaussianRasterizer
    ref = Golden(request)
    P = 40000
    cam, xyz = _straddling_scene(P)
    bg = torch.zeros(3, device="cuda")
    ours = GaussianRasterizer(_settings(cam, bg, 3)).markVisible(xyz)
    assert ours.dtype == torch.bool and ours.shape == (P,)
    assert ref.equal("visible", ours)
    want = ours
    assert 0.2 < float(want.float().mean()) < 0.9                 # the scene really straddles the plane
    # and the rasterizer's own culling agrees with it on the same points: radii > 0 implies visible
    raw = syn.make_gaussians(P, scale_mu=0.02, seed=5, device="cuda")
    act = syn.activated(raw)
    color, radii, depth = GaussianRasterizer(_settings(cam, bg, 3))(
        means3D=xyz, means2D=torch.zeros_like(xyz), opacities=act["opacities"], shs=act["shs"], scales=act["scales"],
        rotations=act["rotations"])
    assert ref.equal("radii", radii)
    assert bool((want | (radii == 0)).all())
    assert ref.maxdiff("color", color) <= COLOR_TOL


def test_prefiltered_flag_is_accepted_when_nothing_is_culled():
    """prefiltered=True promises that no Gaussian fails the frustum test (auxiliary.h:154-162 traps otherwise): with every
    point in front of the camera the outputs equal the prefiltered=False ones bit for bit."""
    from diff_gaussian_rasterization import GaussianRasterizer
    P, W, H = 8000, 128, 80
    raw = syn.make_gaussians(P, scale_mu=0.02, seed=9, device="cuda")
    act = syn.activated(raw)
    cam = syn.make_camera(W, H, device="cuda")
    bg = torch.tensor([0.1, 0.1, 0.1], device="cuda")
    outs = []
    for pre in (False, True):
        outs.append(GaussianRasterizer(_settings(cam, bg, 3, prefiltered=pre))(
            means3D=act["means3D"], means2D=torch.zeros_like(act["means3D"]), opacities=act["opacities"], shs=act["shs"],
            scales=act["scales"], rotations=act["rotations"]))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
