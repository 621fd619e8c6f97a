"""Fused elementwise pieces of the training loop (csrc/elementwise.cu) for b200gs.engine.

The reference spells these with stock PyTorch ops inside code that runs unchanged on top of the
drop-ins (gaussian_renderer/__init__.py:130-132 activations; utils/loss_utils.py:23-24 L1), so they
stay PyTorch there. Our own trainer (`engine.render` / `ViewParallelTrainer`) calls these instead:
one launch each way for exp / normalize / sigmoid, one launch for the loss and its gradient.
The optional D-SSIM term (utils/loss_utils.py:ssim, csrc/ssim.cu) has both forms: `dssim_loss_and_grad` for our trainer and
`ssim`, an autograd drop-in that b200gs.launcher puts in place of the reference's own function.
"""
import ctypes

import torch

from . import _lib
from ._lib import check, current_stream

_P = ctypes.c_void_p
_lib.register("b200gs_activations_forward", ctypes.c_int, [ctypes.c_longlong, _P, _P, _P, _P, _P, _P, _P])
_lib.register("b200gs_activations_backward", ctypes.c_int, [ctypes.c_longlong] + [_P] * 10)
_lib.register("b200gs_l1_loss_fwd_bwd", ctypes.c_int, [ctypes.c_longlong, _P, _P, ctypes.c_float, _P, _P, _P, _P])
_lib.register("b200gs_l1_loss_fwd_bwd_u8", ctypes.c_int, [ctypes.c_int, ctypes.c_int, _P, _P, ctypes.c_float, _P, _P, _P, _P])
_lib.register("b200gs_ssim_scratch_bytes", ctypes.c_size_t, [ctypes.c_int] * 5)
_lib.register("b200gs_ssim_fwd_bwd", ctypes.c_int, [ctypes.c_int] * 4 + [_P, _P, ctypes.c_float, ctypes.c_float, _P, ctypes.c_float, _P, _P,
                                                                       ctypes.c_size_t, _P])
_lib.register("b200gs_ssim_fwd_bwd_u8", ctypes.c_int, [ctypes.c_int, ctypes.c_int, _P, _P, ctypes.c_float, ctypes.c_float, _P,
                                                       ctypes.c_float, _P, _P, ctypes.c_size_t, _P])


def _req(t, shape_tail):
    if not (t.is_cuda and t.dtype == torch.float32):
        raise RuntimeError("fused activations need float32 CUDA tensors (there is no CPU path)")
    if t.dim() != 2 or t.shape[1] != shape_tail:
        raise RuntimeError(f"expected a [P,{shape_tail}] tensor, got {tuple(t.shape)}")
    return t.contiguous()


class _Activations(torch.autograd.Function):
    """(exp(scales), F.normalize(rotations), sigmoid(opacity)) — scene/gaussian_model.py:37-47."""

    @staticmethod
    def forward(ctx, scales, rotations, opacity):
        s, r, o = _req(scales, 3), _req(rotations, 4), _req(opacity, 1)
        P = int(s.shape[0])
        so, ro, oo = torch.empty_like(s), torch.empty_like(r), torch.empty_like(o)
        check(_lib.lib().b200gs_activations_forward(P, s.data_ptr(), r.data_ptr(), o.data_ptr(), so.data_ptr(), ro.data_ptr(),
                                                    oo.data_ptr(), current_stream()), "activations_forward")
        ctx.save_for_backward(so, r, oo)
        return so, ro, oo

    @staticmethod
    def backward(ctx, gs, gr, go):
        so, r, oo = ctx.saved_tensors
        P = int(so.shape[0])
        need = ctx.needs_input_grad
        ds = torch.empty_like(so) if need[0] else None
        dr = torch.empty_like(r) if need[1] else None
        do = torch.empty_like(oo) if need[2] else None
        # contiguous copies of the upstream gradients stay referenced until the launch has been queued
        gs, gr, go = (t.contiguous() if t is not None else None for t in (gs, gr, go))
        p = lambda t: t.data_ptr() if t is not None else None
        check(_lib.lib().b200gs_activations_backward(P, so.data_ptr(), r.data_ptr(), oo.data_ptr(), p(gs), p(gr), p(go),
                                                     p(ds), p(dr), p(do), current_stream()), "activations_backward")
        return ds, dr, do


def activations(scales, rotations, opacity):
    return _Activations.apply(scales, rotations, opacity)


def psnr_from_sse(sse, n):
    """utils/image_utils.py:17-38 from the per-image sums of squared errors the L1 kernel leaves behind:
    20 log10(1 / sqrt(mse)) per image (a device tensor; reading it is the caller's sync)."""
    return 20.0 * torch.log10(1.0 / torch.sqrt(sse / float(n)))


def l1_loss_and_grad(render, target, scale, loss_accum, sse_accum=None):
    """loss_accum[0] += scale * sum|render - target|; returns d(loss)/d(render) (= scale * sign).
    sse_accum (optional, a 1-element float32 CUDA tensor the caller zeroes): += sum (render - target)^2, see psnr_from_sse.
    target: float32 [3,H,W], or the dataset's own uint8 [H,W,3] image (converted on the device as PILtoTorch does: u8 / 255)."""
    sse = None
    if sse_accum is not None:
        if not (sse_accum.is_cuda and sse_accum.dtype == torch.float32 and sse_accum.numel() >= 1):
            raise RuntimeError("l1_loss_and_grad: sse_accum must be a float32 CUDA tensor")
        sse = sse_accum.data_ptr()
    if target.dtype == torch.uint8:
        if not (render.is_cuda and target.is_cuda and render.dtype == torch.float32 and render.dim() == 3 and render.shape[0] == 3
                and tuple(target.shape) == (render.shape[1], render.shape[2], 3)):
            raise RuntimeError("l1_loss_and_grad: a uint8 target must be [H,W,3] on the GPU for a float32 [3,H,W] render")
        r, t = render.detach().contiguous(), target.contiguous()
        d = torch.empty_like(r)
        check(_lib.lib().b200gs_l1_loss_fwd_bwd_u8(int(r.shape[1]), int(r.shape[2]), r.data_ptr(), t.data_ptr(), float(scale),
                                                   loss_accum.data_ptr(), sse, d.data_ptr(), current_stream()), "l1_loss_u8")
        return d
    if not (render.is_cuda and target.is_cuda and render.dtype == torch.float32 and target.dtype == torch.float32):
        raise RuntimeError("l1_loss_and_grad needs float32 CUDA tensors (there is no CPU path)")
    if render.shape != target.shape:
        raise RuntimeError("render / target shape mismatch")
    r, t = render.detach().contiguous(), target.contiguous()
    d = torch.empty_like(r)
    check(_lib.lib().b200gs_l1_loss_fwd_bwd(r.numel(), r.data_ptr(), t.data_ptr(), float(scale), loss_accum.data_ptr(), sse,
                                            d.data_ptr(), current_stream()), "l1_loss")
    return d


def _ssim_launch(x, y, value_offset, value_scale, ssim_sum, weight, d_x):
    """One call of the SSIM kernels (csrc/ssim.cu) on contiguous float32 CUDA x [N,C,H,W] and y (the same, or a uint8 [H,W,3]
    image for a [1,3,H,W] x).  ssim_sum[n] += value_offset + value_scale * sum of image n's map; d_x += weight * d(sum map)/dx
    (d_x None = value only).  The scratch comes from torch's caching allocator."""
    N, C, H, W = (int(s) for s in x.shape)
    L = _lib.lib()
    nbytes = int(L.b200gs_ssim_scratch_bytes(N, C, H, W, int(d_x is not None)))
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    sp = lambda t: t.data_ptr() if t is not None else None
    if y.dtype == torch.uint8:
        check(L.b200gs_ssim_fwd_bwd_u8(H, W, x.data_ptr(), y.data_ptr(), float(value_offset), float(value_scale), sp(ssim_sum),
                                       float(weight), sp(d_x), sp(scratch), nbytes, current_stream()), "ssim_u8")
    else:
        check(L.b200gs_ssim_fwd_bwd(N, C, H, W, x.data_ptr(), y.data_ptr(), float(value_offset), float(value_scale), sp(ssim_sum),
                                    float(weight), sp(d_x), sp(scratch), nbytes, current_stream()), "ssim")


def dssim_loss_and_grad(render, target, weight, loss_accum, d_render):
    """The D-SSIM term of train_4DGS.py for one view: loss_accum[0] += weight * (1 - ssim(render, target)) and
    d_render += weight * d(1 - ssim)/d(render), both in place (d_render is typically what l1_loss_and_grad returned).
    render: float32 [3,H,W] on the GPU; target: float32 [3,H,W], or the dataset's uint8 [H,W,3] image (converted as u8 / 255)."""
    if not (render.is_cuda and render.dtype == torch.float32 and render.dim() == 3 and render.shape[0] == 3):
        raise RuntimeError("dssim_loss_and_grad: render must be a float32 [3,H,W] CUDA tensor (there is no CPU path)")
    if not (loss_accum.is_cuda and loss_accum.dtype == torch.float32 and loss_accum.numel() >= 1):
        raise RuntimeError("dssim_loss_and_grad: loss_accum must be a float32 CUDA tensor")
    if not (d_render.is_cuda and d_render.dtype == torch.float32 and d_render.shape == render.shape and d_render.is_contiguous()):
        raise RuntimeError("dssim_loss_and_grad: d_render must be a contiguous float32 CUDA tensor shaped like render")
    H, W = int(render.shape[1]), int(render.shape[2])
    if target.dtype == torch.uint8:
        if not (target.is_cuda and tuple(target.shape) == (H, W, 3)):
            raise RuntimeError("dssim_loss_and_grad: a uint8 target must be [H,W,3] on the GPU for a [3,H,W] render")
    elif not (target.is_cuda and target.dtype == torch.float32 and target.shape == render.shape):
        raise RuntimeError("dssim_loss_and_grad: target must be float32 [3,H,W] (or uint8 [H,W,3]) on the GPU")
    n = 3 * H * W
    x = render.detach().contiguous().view(1, 3, H, W)
    y = target.contiguous() if target.dtype == torch.uint8 else target.contiguous().view(1, 3, H, W)
    # weight * (1 - sum(map) / n): the constant goes in as the kernel's value offset, -weight / n scales the map sum and its gradient
    _ssim_launch(x, y, weight, -weight / n, loss_accum, -weight / n, d_render)


class _SSIM(torch.autograd.Function):
    """ssim(img1, img2) with the gradient with respect to img1 computed in the forward launch pair (unit weight per image) and
    scaled by grad_output in the backward."""

    @staticmethod
    def forward(ctx, img1, img2, size_average):
        x, y = img1.detach().contiguous(), img2.detach().contiguous()
        if x.dim() == 3:
            x, y = x.unsqueeze(0), y.unsqueeze(0)
        N, C, H, W = (int(s) for s in x.shape)
        per_image = torch.zeros(N, dtype=torch.float32, device=x.device)
        grad = torch.zeros_like(x) if ctx.needs_input_grad[0] else None
        # per_image[n] = mean of image n's map; grad = d(sum_n per_image[n]) / d img1
        _ssim_launch(x, y, 0.0, 1.0 / (C * H * W), per_image, 1.0 / (C * H * W), grad)
        ctx.size_average, ctx.N, ctx.shape = size_average, N, img1.shape
        ctx.save_for_backward(grad)
        if size_average:
            return per_image.mean()
        return per_image if img1.dim() == 4 else per_image.reshape(())

    @staticmethod
    def backward(ctx, grad_output):
        grad, = ctx.saved_tensors
        if grad is None:
            return None, None, None
        if ctx.size_average:
            g = grad * (grad_output / ctx.N)
        else:
            g = grad * grad_output.reshape(-1, 1, 1, 1)
        return g.reshape(ctx.shape), None, None


def ssim(img1, img2, window_size=11, size_average=True):
    """Drop-in for utils/loss_utils.py:ssim on float32 CUDA tensors [N,C,H,W] or [C,H,W] with window_size 11: the map is never
    materialised, its mean and its gradient with respect to img1 come from two launches (csrc/ssim.cu).  size_average=False
    returns one value per image ([N]; a 0-d tensor for a [C,H,W] input).  No gradient flows to img2."""
    if window_size != 11:
        raise RuntimeError("fused ssim: only window_size 11 is implemented")
    if not (img1.is_cuda and img2.is_cuda and img1.dtype == torch.float32 and img2.dtype == torch.float32):
        raise RuntimeError("fused ssim needs float32 CUDA tensors (there is no CPU path)")
    if img1.shape != img2.shape or img1.dim() not in (3, 4) or img1.numel() == 0:
        raise RuntimeError(f"fused ssim: expected two equal [N,C,H,W] or [C,H,W] shapes, got {tuple(img1.shape)} / {tuple(img2.shape)}")
    if img2.requires_grad and torch.is_grad_enabled():
        raise RuntimeError("fused ssim: no gradient with respect to img2")
    return _SSIM.apply(img1, img2, bool(size_average))
