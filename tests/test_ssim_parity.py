"""The fused SSIM / D-SSIM term (csrc/ssim.cu, fusedops.ssim / dssim_loss_and_grad, launcher.patch_loss_utils, the trainer's
lambda_dssim) against the float64 restatement of utils/loss_utils.py:ssim (oracle/ssim_torch.py).

Every GPU check is anchored on float64: PyTorch's own float32 SSIM blurs in TF32 by default (cudnn.allow_tf32), whose
10-bit mantissa already moves s11 = E[x^2] - mu^2 by a few percent of C2, so it is compared only with TF32 off."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import ssim_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------- CPU ---
def _scipy_map(x, y, window):
    """SSIM map of float64 numpy [C,H,W] images with scipy's zero-padded correlation (independent of torch's conv2d)."""
    from scipy.ndimage import correlate
    blur = lambda a: np.stack([correlate(a[c], window, mode="constant", cval=0.0) for c in range(a.shape[0])])
    mu1, mu2 = blur(x), blur(y)
    s11, s22, s12 = blur(x * x) - mu1 ** 2, blur(y * y) - mu2 ** 2, blur(x * y) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    return ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 ** 2 + mu2 ** 2 + C1) * (s11 + s22 + C2))


@pytest.mark.parametrize("shape", [(1, 3, 16, 20), (2, 3, 3, 5), (1, 1, 12, 9), (1, 3, 1, 1)])
def test_oracle_matches_scipy_correlate(shape):
    g = torch.Generator().manual_seed(7)
    x = torch.rand(shape, generator=g, dtype=torch.float64)
    y = (x + 0.2 * torch.rand(shape, generator=g, dtype=torch.float64)).clamp(0, 1)
    ours = ssim_torch.ssim_map(x, y).numpy()
    window = ssim_torch.create_window(11, 1)[0, 0].double().numpy()
    for n in range(shape[0]):
        ref = _scipy_map(x[n].numpy(), y[n].numpy(), window)
        np.testing.assert_allclose(ours[n], ref, rtol=1e-12, atol=1e-12)
    per_image = ssim_torch.ssim(x, y, size_average=False)
    assert per_image.shape == (shape[0],)
    assert torch.allclose(ssim_torch.ssim(x, y), per_image.mean(), rtol=1e-14, atol=0)


def test_oracle_window_is_the_reference_gaussian():
    from math import exp
    g = ssim_torch.gaussian(11, 1.5)
    assert g.dtype == torch.float32 and abs(float(g.sum()) - 1.0) < 1e-6
    raw = np.array([exp(-(x - 5) ** 2 / 4.5) for x in range(11)], dtype=np.float32)
    np.testing.assert_allclose(g.numpy(), raw / raw.sum(dtype=np.float32), rtol=2e-7)
    w = ssim_torch.create_window(11, 3)
    assert w.shape == (3, 1, 11, 11) and w.dtype == torch.float32 and torch.equal(w[0, 0], w[0, 0].t())


def test_oracle_gradcheck():
    g = torch.Generator().manual_seed(3)
    x = torch.rand(2, 3, 9, 13, generator=g, dtype=torch.float64, requires_grad=True)
    y = torch.rand(2, 3, 9, 13, generator=g, dtype=torch.float64)
    assert torch.autograd.gradcheck(lambda a: ssim_torch.ssim(a, y), (x,), eps=1e-6, atol=1e-8, rtol=1e-6)
    assert torch.autograd.gradcheck(lambda a: ssim_torch.ssim(a, y, size_average=False), (x,), eps=1e-6, atol=1e-8, rtol=1e-6)


def _closed_form(x, y):
    """The kernels' algorithm in float64 numpy: separable 11-tap blurs, the map, A / B / Cc, three more blurs."""
    g = ssim_torch.gaussian(11, 1.5).double().numpy()

    def blur(a):                                   # [C,H,W], zero padding, correlation (= convolution: g is symmetric)
        C, H, W = a.shape
        p = np.zeros((C, H + 10, W + 10)); p[:, 5:5 + H, 5:5 + W] = a
        h = sum(g[k] * p[:, :, k:k + W] for k in range(11))
        return sum(g[k] * h[:, k:k + H, :] for k in range(11))
    mu1, mu2 = blur(x), blur(y)
    s11, s22, s12 = blur(x * x) - mu1 ** 2, blur(y * y) - mu2 ** 2, blur(x * y) - mu1 * mu2
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    n1, n2, d1, d2 = 2 * mu1 * mu2 + C1, 2 * s12 + C2, mu1 ** 2 + mu2 ** 2 + C1, s11 + s22 + C2
    m = n1 * n2 / (d1 * d2)
    B = -m / d2
    Cc = 2 * n1 / (d1 * d2)
    A = 2 * mu2 * n2 / (d1 * d2) - 2 * mu1 * m / d1 - 2 * mu1 * B - mu2 * Cc
    return m, blur(A) + 2 * x * blur(B) + y * blur(Cc)


@pytest.mark.parametrize("shape", [(3, 17, 23), (1, 4, 6), (3, 40, 33)])
def test_closed_form_gradient_matches_oracle_autograd(shape):
    """The backward the kernels implement (dL/dx = w*A + 2x w*B + y w*Cc for L = sum map) is autograd's gradient."""
    g = torch.Generator().manual_seed(11)
    x = torch.rand(shape, generator=g, dtype=torch.float64)
    y = torch.rand(shape, generator=g, dtype=torch.float64)
    m, grad = _closed_form(x.numpy(), y.numpy())
    per_image, ref = ssim_torch.ssim_and_grad(x[None], y[None])
    # the reference's 2-D window is the float32-ROUNDED outer product g g^T, the separable blur applies g_i g_j exactly:
    # the two differ by one float32 rounding per weight (~6e-8 relative), nothing else
    np.testing.assert_allclose(m.mean(), float(per_image[0]), rtol=5e-7)
    np.testing.assert_allclose(grad, ref[0].numpy(), rtol=0, atol=2e-6 * np.abs(ref.numpy()).max())


class _FakeCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so that the routing predicate can be exercised without a GPU."""
    @property
    def is_cuda(self):
        return True


def _stand_in_module():
    calls = []
    mod = types.ModuleType("loss_utils_stand_in")

    def ssim(img1, img2, window_size=11, size_average=True):
        calls.append((window_size, size_average))
        return "original"
    mod.ssim = ssim
    return mod, calls


def test_patch_loss_utils_routing(monkeypatch):
    from b200gs import fusedops, launcher
    monkeypatch.delenv("B200GS_FUSED_SSIM", raising=False)
    fused_calls = []
    monkeypatch.setattr(fusedops, "ssim", lambda a, b, w=11, s=True: fused_calls.append((w, s)) or "fused")
    mod, calls = _stand_in_module()
    orig = mod.ssim
    launcher.patch_loss_utils(mod)
    launcher.patch_loss_utils(mod)                       # idempotent: wraps once
    assert mod.ssim is not orig and mod.ssim._b200gs_original is orig

    a, b = torch.rand(2, 3, 20, 24), torch.rand(2, 3, 20, 24)
    fa, fb = a.as_subclass(_FakeCuda), b.as_subclass(_FakeCuda)
    sup = launcher.fused_ssim_supported
    assert sup(fa, fb) and sup(fa, fb, 11, False) and sup(fa[0], fb[0])
    assert not sup(a, b)                                 # CPU tensors
    assert not sup(fa, fb, 7)                            # another window
    assert not sup(fa.double(), fb.double())             # not float32
    assert not sup(fa, fb[:, :, :10])                    # shapes differ
    assert not sup(fa[0], fb[0], 11, False)              # [C,H,W] with size_average=False: the reference's own error
    fb_grad = b.clone().requires_grad_(True).as_subclass(_FakeCuda)
    assert not sup(fa, fb_grad)                          # a gradient for img2
    with torch.no_grad():
        assert sup(fa, fb_grad)                          # ... unless autograd is off

    # supported calls go to fusedops.ssim, everything else to the original
    assert mod.ssim(fa, fb) == "fused" and fused_calls == [(11, True)]
    assert mod.ssim(fa, fb, 11, False) == "fused" and fused_calls[-1] == (11, False)
    assert mod.ssim(a, b) == "original"
    assert mod.ssim(fa, fb, window_size=7) == "original" and calls[-1] == (7, True)
    assert mod.ssim(fa, fb_grad) == "original"
    assert len(calls) == 3 and len(fused_calls) == 2


def test_patch_loss_utils_disabled_by_environment(monkeypatch):
    from b200gs import launcher
    monkeypatch.setenv("B200GS_FUSED_SSIM", "0")
    mod, _ = _stand_in_module()
    orig = mod.ssim
    assert launcher.patch_loss_utils(mod) is mod and mod.ssim is orig


class _TinyModel(torch.nn.Module):
    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self._xyz = torch.nn.Parameter(torch.randn(20, 3, generator=g))
        self._opacity = torch.nn.Parameter(torch.randn(20, 1, generator=g))
        self.optimizer = torch.optim.Adam(self.parameters(), lr=1e-3)

    @property
    def get_xyz(self):
        return self._xyz


def _tiny_render(cam, model, bg, stage):
    sp = torch.zeros_like(model._xyz, requires_grad=True)
    v = (torch.sigmoid(model._opacity) * (model._xyz + sp)).sum() * cam
    img = v * torch.ones(3, 12, 14) + bg[:, None, None]
    return {"render": img, "viewspace_points": sp, "radii": torch.zeros(20, dtype=torch.int32)}


def test_trainer_plain_path_refuses_dssim():
    from b200gs.engine import ViewParallelTrainer, default_opt
    assert default_opt().lambda_dssim == 0.0
    gts = [torch.rand(3, 12, 14) for _ in range(2)]
    tr = ViewParallelTrainer(_TinyModel(), torch.zeros(3), stage="fine", render_fn=_tiny_render, lambda_dssim=0.2)
    with pytest.raises(NotImplementedError):
        tr.step([0.5, 0.7], gts)
    # lambda_dssim = 0 is the plain L1 path as before
    tr0 = ViewParallelTrainer(_TinyModel(), torch.zeros(3), stage="fine", render_fn=_tiny_render)
    assert torch.isfinite(tr0.step([0.5, 0.7], gts))


# ---------------------------------------------------------------------------------------------------------------- GPU ---
SHAPES = [(1, 3, 720, 1280), (2, 3, 37, 53), (1, 3, 5, 7), (1, 1, 64, 64), (1, 3, 1080, 1920)]
KINDS = ["independent", "perturbed", "constant"]


def _inputs(shape, kind, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "independent":
        return (torch.rand(shape, device="cuda", generator=g), torch.rand(shape, device="cuda", generator=g))
    if kind == "perturbed":
        y = torch.rand(shape, device="cuda", generator=g)
        return (y + 0.01 * torch.randn(shape, device="cuda", generator=g)).clamp(0, 1), y
    return torch.full(shape, 0.3, device="cuda"), torch.full(shape, 0.7, device="cuda")


def _fused(x, y, weight=1.0, d_x=None, grad=True):
    from b200gs import fusedops
    sums = torch.zeros(x.shape[0], device=x.device)
    if grad and d_x is None:
        d_x = torch.zeros_like(x)
    fusedops._ssim_launch(x, y, 0.0, 1.0, sums, weight, d_x if grad else None)
    return sums, d_x


def _check_grad(g, g64, what=""):
    """max |g - g64| <= 1e-4 max |g64|; per element <= 1e-3 relative wherever |g64| >= 1e-2 max |g64|."""
    g64 = g64.double()
    err = (g.double() - g64).abs()
    gmax = float(g64.abs().max())
    if gmax == 0.0:
        assert float(err.max()) <= 1e-6, what
        return
    assert float(err.max()) <= 1e-4 * gmax, (what, float(err.max()) / gmax)
    big = g64.abs() >= 1e-2 * gmax
    rel = float((err[big] / g64.abs()[big]).max())
    assert rel <= 1e-3, (what, rel)


@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_value_and_gradient_against_float64(shape, kind):
    x, y = _inputs(shape, kind)
    sums, d = _fused(x, y)
    per_image64, g64 = ssim_torch.ssim_and_grad(x, y)
    n = shape[1] * shape[2] * shape[3]
    sums64 = per_image64 * n
    assert float(((sums.double() - sums64).abs() / sums64.abs().clamp_min(1e-30)).max()) <= 1e-5, (sums, sums64)
    assert abs(float(sums.double().sum()) / (n * shape[0]) - float(per_image64.mean())) <= 2e-6
    _check_grad(d, g64, (shape, kind))


@gpu
def test_gradient_is_added_and_value_only_call_writes_nothing():
    x, y = _inputs((2, 3, 150, 203), "independent", seed=5)
    _, d_null = _fused(x, y, weight=0.37)
    prior = torch.randn_like(x)
    _, d_acc = _fused(x, y, weight=0.37, d_x=prior.clone())
    # prior + (0.37 * g), one FP32 add (the kernel may contract the multiply into it: then within one rounding of the add)
    tol = torch.finfo(torch.float32).eps * (prior.abs() + d_null.abs())
    assert bool(((d_acc - (prior + d_null)).abs() <= tol).all())
    xs, ys = x.clone(), y.clone()
    sums_v, none = _fused(x, y, grad=False)
    sums_g, _ = _fused(x, y)
    assert none is None and torch.equal(x, xs) and torch.equal(y, ys)
    assert torch.allclose(sums_v, sums_g, rtol=1e-6, atol=0)


@gpu
@pytest.mark.parametrize("H,W", [(720, 1280), (37, 53), (5, 7)])
def test_uint8_target_equals_float_path(H, W):
    """The uint8 [H,W,3] target converted on the device (u8 / 255) gives BITWISE the float path's gradient; the per-image sums
    agree to the order of the CTAs' FP64 atomic adds: within 1 ULP of the FP32 result."""
    from b200gs import fusedops
    g = torch.Generator(device="cuda").manual_seed(2)
    u8 = torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    x = torch.rand(1, 3, H, W, device="cuda", generator=g)
    # PILtoTorch divides on the host (IEEE division); torch's CUDA division by a scalar multiplies by the reciprocal instead
    yf = (u8.cpu().permute(2, 0, 1).float() / 255).unsqueeze(0).contiguous().cuda()
    sf, df = _fused(x, yf, weight=0.5)
    su, du = _fused(x, u8, weight=0.5)
    assert torch.equal(du, df)
    assert float((su - sf).abs().max()) <= float(torch.finfo(torch.float32).eps * sf.abs().max()), (su, sf)
    # the trainer's form: both accumulators in place
    lf, lu = torch.full((1,), 0.25, device="cuda"), torch.full((1,), 0.25, device="cuda")
    df2, du2 = torch.ones_like(x[0]), torch.ones_like(x[0])
    fusedops.dssim_loss_and_grad(x[0], yf[0], 0.2, lf, df2)
    fusedops.dssim_loss_and_grad(x[0], u8, 0.2, lu, du2)
    assert torch.equal(du2, df2) and float((lu - lf).abs()) <= float(torch.finfo(torch.float32).eps * lf.abs())


@gpu
def test_dssim_loss_and_grad_against_float64():
    from b200gs import fusedops
    x, y = _inputs((1, 3, 91, 130), "independent", seed=9)
    w = 0.3
    loss = torch.full((1,), 0.5, device="cuda")
    d = torch.zeros_like(x[0])             # (adding into a non-zero buffer: test_gradient_is_added_and_value_only_call_writes_nothing)
    fusedops.dssim_loss_and_grad(x[0], y[0], w, loss, d)
    per_image64, g64 = ssim_torch.ssim_and_grad(x, y)
    n = x.numel()
    assert abs(float(loss) - (0.5 + w * (1 - float(per_image64[0])))) <= 2e-6
    _check_grad(d, -w / n * g64[0], "dssim")


@gpu
@pytest.mark.parametrize("shape", [(2, 3, 64, 80), (3, 48, 50)], ids=["NCHW", "CHW"])
@pytest.mark.parametrize("size_average", [True, False])
def test_dropin_ssim_against_float64(shape, size_average):
    from b200gs import fusedops
    g = torch.Generator(device="cuda").manual_seed(4)
    a = torch.rand(shape, device="cuda", generator=g)
    b = (a + 0.1 * torch.rand(shape, device="cuda", generator=g)).clamp(0, 1)
    x = a.clone().requires_grad_(True)
    out = fusedops.ssim(x, b, 11, size_average)
    x64 = a.double().requires_grad_(True)
    ref = ssim_torch.ssim(x64, b.double(), 11, size_average) if (size_average or len(shape) == 4) else \
        ssim_torch.ssim(x64[None], b.double()[None], 11, False)[0]
    assert out.shape == ref.shape and out.dtype == torch.float32
    assert float((out.detach().double() - ref.detach()).abs().max()) <= 2e-6
    go = torch.rand(ref.shape, device="cuda", dtype=torch.float64, generator=g) * 3 - 1 if ref.dim() else torch.tensor(-2.5, device="cuda", dtype=torch.float64)
    out.backward(go.float())
    ref.backward(go)
    _check_grad(x.grad, x64.grad, "dropin")
    # PyTorch's float32 SSIM with TF32 off lands within the same bars (with TF32 on it does not: see the module docstring)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        x32 = a.clone().requires_grad_(True)
        r32 = ssim_torch.ssim(x32, b, 11, size_average) if (size_average or len(shape) == 4) else \
            ssim_torch.ssim(x32[None], b[None], 11, False)[0]
        r32.backward(go.float())
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert float((r32.double() - ref.detach()).abs().max()) <= 2e-6
    _check_grad(x32.grad, x64.grad, "torch fp32, tf32 off")
    # no gradient wanted: value only
    with torch.no_grad():
        assert torch.allclose(fusedops.ssim(a, b, 11, size_average), out.detach(), rtol=1e-6, atol=0)


@gpu
def test_trainer_lambda_zero_takes_todays_path(monkeypatch):
    from b200gs import engine, fusedops, synthetic as syn
    tr, cams, gts = _small_scene(lambda_dssim=0.0)

    def boom(*a, **k):
        raise AssertionError("dssim_loss_and_grad must not run with lambda_dssim = 0")
    monkeypatch.setattr(fusedops, "dssim_loss_and_grad", boom)
    assert torch.isfinite(tr.step(cams, gts))


def _small_scene(lambda_dssim):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    P, W, H = 30000, 240, 144
    raw = syn.make_gaussians(P, scale_mu=0.012, seed=3, device="cpu")
    torch.manual_seed(0)
    m = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}).to(dev)
    m.training_setup()
    tr = engine.ViewParallelTrainer(m, torch.tensor([0.05, 0.1, 0.15], device=dev), stage="fine", lambda_dssim=lambda_dssim)
    cams = syn.orbit_cameras(2, W, H, device=dev)
    g = torch.Generator().manual_seed(1)
    gts = [torch.rand(3, H, W, generator=g).to(dev) for _ in cams]
    return tr, cams, gts


@gpu
def test_trainer_lambda_dssim_loss_and_image_gradient(monkeypatch):
    from b200gs import fusedops
    lam = 0.2
    tr, cams, gts = _small_scene(lambda_dssim=lam)
    seen = []
    real = fusedops.dssim_loss_and_grad

    def spy(render, target, weight, loss_accum, d_render):
        real(render, target, weight, loss_accum, d_render)
        seen.append((render.detach().clone(), target.clone(), weight, d_render.detach().clone()))
    monkeypatch.setattr(fusedops, "dssim_loss_and_grad", spy)
    loss = float(tr.step(cams, gts))
    B = len(cams)
    assert len(seen) == B and all(abs(w - lam / B) < 1e-12 for _, _, w, _ in seen)
    want = 0.0
    for img, gt, _, d in seen:
        x, y = img.double(), gt.double()
        n = x.numel()
        per_image64, g64 = ssim_torch.ssim_and_grad(img[None], gt[None])
        want += float((x - y).abs().mean()) / B + lam / B * (1.0 - float(per_image64[0]))
        d64 = torch.sign(x - y) / (n * B) - lam / B / n * g64[0]
        _check_grad(d, d64, "trainer image gradient")
    assert abs(loss - want) <= 1e-5 * abs(want), (loss, want)


REF = os.path.join(ROOT, "baseline", "_ref")


@gpu
@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "utils", "loss_utils.py")), reason="baseline/_ref not installed")
def test_reference_ssim_with_tf32_off_matches_dropin():
    import importlib.util
    from b200gs import fusedops
    spec = importlib.util.spec_from_file_location("ref_loss_utils", os.path.join(REF, "utils", "loss_utils.py"))
    saved = list(sys.path)
    sys.path.insert(0, REF)
    try:
        lu = importlib.util.module_from_spec(spec); spec.loader.exec_module(lu)
    finally:
        sys.path[:] = saved
    g = torch.Generator(device="cuda").manual_seed(8)
    a = torch.rand(2, 3, 90, 120, device="cuda", generator=g)
    b = (a + 0.1 * torch.rand(a.shape, device="cuda", generator=g)).clamp(0, 1)
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        xr = a.clone().requires_grad_(True)
        r = lu.ssim(xr, b)
        r.backward()
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    xf = a.clone().requires_grad_(True)
    f = fusedops.ssim(xf, b)
    f.backward()
    assert abs(float(f) - float(r)) <= 2e-6
    _check_grad(xf.grad, xr.grad, "reference fp32")
