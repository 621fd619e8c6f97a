"""Drop-in HexPlane deformation field: `HexPlaneField`, `Deformation`, `deform_network`.

Mirrors scene/hexplane.py:109-183 and scene/deformation.py:16-242 — same constructor
arguments, attribute paths, parameter names / shapes (so `state_dict()` keys such as
`deformation_net.grid.grids.{level}.{plane}`, `deformation_net.grid.aabb`,
`deformation_net.feature_out.0.weight`, `timenet.*`, `*_poc` match), same call signatures and
return values — while forward and backward run the hand-written sm_100a kernels of
libb200gs (csrc/hexplane.cu, csrc/deform_mlp*.cu and, with `no_do` / `no_dshs` False, csrc/deform_heads.cu for the
opacity and SH heads) through `torch.autograd.Function`s.

Differences that do not change results:
  * plane parameters keep their [1, C, H, W] shape (C = 16 or 32) but use torch.channels_last strides
    (one coalesced line of C floats per texel in the kernels);
  * the sin/cos positional encodings the reference computes and then slices away
    (deformation.py:205-207 vs :107-135) are not computed.
Configurations the reference can express but does not train with are rejected loudly
(NotImplementedError) instead of silently falling back to PyTorch operators.  `HexPlaneField` takes 16 or 32 channels at
1-4 levels; `Deformation` (the fused MLP) needs 32 channels at 2 or 4 levels.  `HexPlaneField` alone can therefore serve
as the grid of the reference's own `scene.deformation.Deformation` (b200gs.launcher.patch_hexplane).
"""
import contextlib
import ctypes
import itertools
import os

import torch
import torch.nn as nn
import torch.nn.init as init

from . import _lib
from ._lib import check, current_stream

MAX_LEVELS = 4


class _HexDesc(ctypes.Structure):
    _fields_ = [("levels", ctypes.c_int), ("channels", ctypes.c_int), ("res", (ctypes.c_int * 4) * MAX_LEVELS),
                ("plane", (ctypes.c_void_p * 6) * MAX_LEVELS), ("grad_plane", (ctypes.c_void_p * 6) * MAX_LEVELS),
                ("aabb", ctypes.c_void_p)]


class _MlpWeights(ctypes.Structure):
    _fields_ = [("feat_dim", ctypes.c_int), ("width", ctypes.c_int), ("w1", ctypes.c_void_p), ("b1", ctypes.c_void_p),
                ("w2", ctypes.c_void_p * 3), ("b2", ctypes.c_void_p * 3), ("w3", ctypes.c_void_p * 3),
                ("b3", ctypes.c_void_p * 3), ("feat_tiled", ctypes.c_int)]


class _MlpGrads(ctypes.Structure):
    _fields_ = [("w1", ctypes.c_void_p), ("b1", ctypes.c_void_p), ("w2", ctypes.c_void_p * 3),
                ("b2", ctypes.c_void_p * 3), ("w3", ctypes.c_void_p * 3), ("b3", ctypes.c_void_p * 3)]


class _HeadsWeights(ctypes.Structure):
    _fields_ = [("feat_dim", ctypes.c_int), ("width", ctypes.c_int), ("w1", ctypes.c_void_p), ("w2", ctypes.c_void_p * 2),
                ("b2", ctypes.c_void_p * 2), ("w3", ctypes.c_void_p * 2), ("b3", ctypes.c_void_p * 2), ("feat_tiled", ctypes.c_int)]


class _HeadsGrads(ctypes.Structure):
    _fields_ = [("w1", ctypes.c_void_p), ("b1", ctypes.c_void_p), ("w2", ctypes.c_void_p * 2),
                ("b2", ctypes.c_void_p * 2), ("w3", ctypes.c_void_p * 2), ("b3", ctypes.c_void_p * 2)]


_P = ctypes.c_void_p
_lib.register("b200gs_hexplane_forward", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, _P, ctypes.c_float, _P, _P])
_lib.register("b200gs_hexplane_backward", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, _P, ctypes.c_float, _P, _P, _P])
_lib.register("b200gs_hexplane_forward_masked", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, _P, ctypes.c_float, ctypes.c_int, _P, _P, _P])
_lib.register("b200gs_hexplane_backward_masked", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, _P, ctypes.c_float, ctypes.c_int, _P, _P, _P, _P, _P, ctypes.c_size_t, _P])
_lib.register("b200gs_hexplane_time_row_scratch_bytes", ctypes.c_size_t, [ctypes.POINTER(_HexDesc), ctypes.c_int])
_lib.register("b200gs_hexplane_time_supported", ctypes.c_int, [ctypes.POINTER(_HexDesc)])
_lib.register("b200gs_hexplane_time_forward", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, ctypes.c_float, _P, _P, ctypes.c_int, _P])
_lib.register("b200gs_hexplane_time_backward", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_longlong, _P, _P, ctypes.c_float, _P, _P, _P, _P, _P, ctypes.c_size_t, ctypes.c_int, _P])
_lib.register("b200gs_hexplane_order_scratch_bytes", ctypes.c_size_t, [ctypes.c_longlong])
_lib.register("b200gs_hexplane_order", ctypes.c_int, [ctypes.c_longlong, _P, _P, _P, _P, ctypes.c_size_t, _P])
_lib.register("b200gs_hexplane_regulation", ctypes.c_int,
              [ctypes.POINTER(_HexDesc), ctypes.c_float, ctypes.c_float, ctypes.c_float, _P, _P])
_lib.register("b200gs_uniform_value", ctypes.c_int, [ctypes.c_longlong, _P, _P, _P, _P])
_lib.register("b200gs_deform_mlp_saved_floats", ctypes.c_size_t, [ctypes.c_longlong])
_lib.register("b200gs_deform_mlp_forward", ctypes.c_int,
              [ctypes.POINTER(_MlpWeights), ctypes.c_longlong, _P, _P, _P, _P, _P, ctypes.c_float, _P, ctypes.c_float,
               _P, _P, _P, _P, _P])
_lib.register("b200gs_deform_mlp_backward", ctypes.c_int,
              [ctypes.POINTER(_MlpWeights), ctypes.POINTER(_MlpGrads), ctypes.c_longlong, _P, _P, _P, _P, _P, _P, _P])
_lib.register("b200gs_deform_heads_saved_floats", ctypes.c_size_t, [ctypes.c_longlong])
_lib.register("b200gs_deform_heads_forward", ctypes.c_int,
              [ctypes.POINTER(_HeadsWeights), ctypes.c_longlong, ctypes.c_int, _P, _P, _P, _P, _P, _P, _P])
_lib.register("b200gs_deform_heads_backward", ctypes.c_int,
              [ctypes.POINTER(_HeadsWeights), ctypes.POINTER(_HeadsGrads), ctypes.c_longlong, ctypes.c_int, _P, _P, _P, _P, _P, _P,
               _P, ctypes.c_int, _P])

_ROW_SCRATCH = {}
TIME_ROW_REPLICAS = 64


def _time_row_scratch(d, device):
    """Scratch for the uniform-timestamp time-plane reduction (b200gs_hexplane_backward_masked), cached per device."""
    n = _lib.lib().b200gs_hexplane_time_row_scratch_bytes(ctypes.byref(d), TIME_ROW_REPLICAS)
    t = _ROW_SCRATCH.get(device)
    if t is None or t.numel() < n:
        t = torch.empty((n,), dtype=torch.uint8, device=device)
        _ROW_SCRATCH[device] = t
    return t, n


_ORDER_CACHE = {}
ORDER_MIN_POINTS = 1 << 14
ORDER_MAX_AGE = 64          # optimiser steps (version bumps of xyz) a cached order is kept for


def _cell_order(pts, aabb):
    """Cell-sorted visiting order of the query points (a locality HINT for the sampling kernels: any permutation gives the
    same results).  Cached per device on the storage: within one training iteration every view and the backward pass query
    the same positions, and across iterations the Gaussians move by a small fraction of a cell, so the order is re-sorted
    only every ORDER_MAX_AGE parameter updates (FusedAdam bumps `_version` per step) or when the tensor / aabb changes.
    The entry holds the tensor it was sorted for: while it lives, its memory cannot be handed to a different tensor, so an
    address match always means the same points.  A per-call copy (the `pts.contiguous()` of the [:, :3] slice the reference's
    Deformation passes) is therefore sorted on every call; a freed copy's recycled address, at version 0, must not pass for
    the same points."""
    P = int(pts.shape[0])
    if P < ORDER_MIN_POINTS:
        return None
    key = (pts.data_ptr(), P, aabb.data_ptr(), aabb._version)
    hit = _ORDER_CACHE.get(pts.device)
    if hit is not None and hit[0] == key and 0 <= pts._version - hit[2] < ORDER_MAX_AGE:
        return hit[1]
    L = _lib.lib()
    order = torch.empty((P,), dtype=torch.int32, device=pts.device)
    nbytes = L.b200gs_hexplane_order_scratch_bytes(P)
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device=pts.device)
    check(L.b200gs_hexplane_order(P, pts.data_ptr(), aabb.data_ptr(), order.data_ptr(), scratch.data_ptr(), nbytes,
                                  current_stream()), "hexplane_order")
    _lib.COUNTERS["cell_order_sorts"] += 1
    _ORDER_CACHE[pts.device] = (key, order, pts._version, pts)
    return order


def _cl(t):
    """[1,C,H,W] tensor in channels_last memory (values unchanged)."""
    return t if t.is_contiguous(memory_format=torch.channels_last) and t.stride(1) == 1 \
        else t.contiguous(memory_format=torch.channels_last)


def _hex_desc(aabb, planes, levels, res, grads=None):
    d = _HexDesc()
    d.levels = levels
    d.channels = int(planes[0].shape[1])
    for l in range(levels):
        for a in range(4):
            d.res[l][a] = int(res[l][a])
        for k in range(6):
            p = planes[l * 6 + k]
            if p.stride(1) != 1:
                raise RuntimeError("HexPlane planes must be channels_last")
            d.plane[l][k] = p.data_ptr()
            d.grad_plane[l][k] = grads[l * 6 + k].data_ptr() if grads is not None and grads[l * 6 + k] is not None else None
    d.aabb = aabb.data_ptr()
    return d


def _check_cuda_f32(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("the B200 deformation field runs on CUDA tensors only (no CPU path)")
        if t.dtype != torch.float32:
            raise RuntimeError(f"expected float32, got {t.dtype}")


# The reference's render() repeats the camera's ONE timestamp into a [P,1] tensor (gaussian_renderer/__init__.py:56).  With this
# switch on (default) a tensor timestamp is checked on the device -- one tiny kernel + an 8-byte read-back, i.e. a host sync a few
# hundred microseconds before the one the rasterizer forward performs anyway -- and a uniform one takes the same one-timestamp
# path as a Python float: time planes served from shared memory, their gradient reduced through 1-D rows.
DETECT_UNIFORM_TIME = os.environ.get("B200GS_DETECT_UNIFORM_TIME", "1") != "0"
_UNIFORM_BUF = {}


def _uniform_time(t):
    """t: contiguous float32 CUDA tensor -> its single value as a Python float if every element is bit-identical, else None."""
    import struct
    buf = _UNIFORM_BUF.get(t.device)
    if buf is None:
        buf = (torch.empty(2, dtype=torch.int32, device=t.device), torch.empty(2, dtype=torch.int32).pin_memory())
        _UNIFORM_BUF[t.device] = buf
    check(_lib.lib().b200gs_uniform_value(t.numel(), t.data_ptr(), buf[0].data_ptr(), buf[1].data_ptr(), current_stream()), "uniform_value")
    if int(buf[1][0]) != 1:
        return None
    return struct.unpack("<f", struct.pack("<I", int(buf[1][1]) & 0xFFFFFFFF))[0]


def _times_arg(times, P, detect=True):
    """times_sel is a [P,1] tensor in the reference (gaussian_renderer/__init__.py:56).  Returns (per-point tensor or None, scalar)."""
    if torch.is_tensor(times):
        t = times.reshape(-1)
        if t.numel() == 1 and P != 1:
            t = t.expand(P)
        if t.numel() != P:
            raise RuntimeError("timestamps must have one entry per point")
        t = t.to(torch.float32).contiguous()
        if detect and DETECT_UNIFORM_TIME and t.is_cuda and P > 0:
            v = _uniform_time(t)
            if v is not None:
                return None, v
        return t, 0.0
    return None, float(times)


class _HexPlaneFn(torch.autograd.Function):
    """features = HexPlaneField(pts, t); inputs (pts, times, aabb, levels, res, *planes)."""

    @staticmethod
    def forward(ctx, pts, times, aabb, levels, res, *planes):
        pts = pts.contiguous()
        _check_cuda_f32(pts, aabb, *planes)
        P = int(pts.shape[0])
        tt, ts = _times_arg(times, P)
        feat = torch.empty((P, int(planes[0].shape[1]) * levels), dtype=torch.float32, device=pts.device)
        d = _hex_desc(aabb, planes, levels, res)
        order = _cell_order(pts, aabb)
        check(_lib.lib().b200gs_hexplane_forward(ctypes.byref(d), P, pts.data_ptr(), _lib.ptr(order),
                                                 tt.data_ptr() if tt is not None else None, ts, feat.data_ptr(),
                                                 current_stream()), "hexplane_forward")
        ctx.save_for_backward(pts, tt if tt is not None else torch.empty(0), aabb, *planes)
        ctx.meta = (levels, res, ts, tt is not None)
        ctx.order = order
        return feat

    @staticmethod
    def backward(ctx, d_feat):
        pts, tt, aabb, *planes = ctx.saved_tensors
        levels, res, ts, has_t = ctx.meta
        P = int(pts.shape[0])
        need_planes = [ctx.needs_input_grad[5 + i] for i in range(len(planes))]
        grads = [torch.zeros_like(p, memory_format=torch.preserve_format) if n else None for p, n in zip(planes, need_planes)]
        d_pts = torch.empty_like(pts) if ctx.needs_input_grad[0] else None
        d = _hex_desc(aabb, planes, levels, res, grads)
        d_feat = d_feat.contiguous()          # kept alive in this frame until the launch has been queued
        if d.channels == 16 and not has_t:
            # One timestamp for the whole call (the reference's render() passes the camera's one time): every point adds into
            # the same two rows of each time plane, so their gradient is reduced through replicated 1-D rows first.
            scratch, nbytes = _time_row_scratch(d, pts.device)
            check(_lib.lib().b200gs_hexplane_backward_masked(ctypes.byref(d), P, pts.data_ptr(), _lib.ptr(ctx.order), None, ts, MASK_ALL,
                                                             None, None, d_feat.data_ptr(),
                                                             d_pts.data_ptr() if d_pts is not None else None, scratch.data_ptr(),
                                                             nbytes, current_stream()), "hexplane_backward")
            return (d_pts, None, None, None, None, *grads)
        check(_lib.lib().b200gs_hexplane_backward(ctypes.byref(d), P, pts.data_ptr(), _lib.ptr(ctx.order),
                                                  tt.data_ptr() if has_t else None, ts, d_feat.data_ptr(),
                                                  d_pts.data_ptr() if d_pts is not None else None, current_stream()),
              "hexplane_backward")
        return (d_pts, None, None, None, None, *grads)


# When True (set by b200gs.engine.ViewParallelTrainer around its views), the backward kernels accumulate the
# weight / plane gradients straight into the parameters' existing `.grad` buffers (the kernels add atomically
# anyway) and autograd gets None for them: per view this saves a zero-fill plus an accumulation pass for each of
# the 26 field parameters. Off by default, so under the reference's own scripts autograd sees ordinary gradients.
ACCUMULATE_INTO_GRAD = False
# Optional callable invoked right after the deformation-MLP backward kernel of a view has been queued (the trainer starts the SH
# gradient's side-stream all-reduce + Adam there on the last view of a step); None = nothing.
AFTER_MLP_BACKWARD = None
# Set by the trainer for the duration of a view when the SH head is on: the [P,16,3] buffer the step's SH gradient collects in.
# The heads backward adds d shs (= d shs', the identity path) into it -- writes it when SH_GRAD_OVERWRITE, the step's first
# view -- and autograd gets None for `shs`.  None = the gradient goes to autograd.
SH_GRAD_ACCUMULATOR = None
SH_GRAD_OVERWRITE = False


def _grad_target(param):
    g = param.grad
    if ACCUMULATE_INTO_GRAD and g is not None and g.dtype == torch.float32 and g.shape == param.shape \
            and g.stride() == param.stride() and g.device == param.device:
        return g
    return None


# ---- the spatial product, shared by several field calls ----------------------------------------------
# The Gaussians' xyz do not change between the views of a batch, so the product of the three SPATIAL planes
# (xy, xz, yz) is the same for every view: b200gs.engine.ViewParallelTrainer evaluates it once per step
# (begin_shared_step), each view then samples only the three TIME planes and multiplies, each view's backward
# accumulates the spatial product's upstream gradient, and ONE spatial backward per step (finish_shared_step)
# scatters it. Same mathematics as six planes per view (the product is re-associated), ~half the gathers / REDs.
# Three holders keep a _SpatialProduct, each for its own lifetime: the explicit scope (_SHARED), the no-grad cache (_INFER), autograd's (_AUTO).
MASK_SPATIAL, MASK_TIME, MASK_ALL = 0x0B, 0x34, 0x3F


def _is_spatial(k):
    """Whether plane k of the planes list (six per level: xy, xz, xt, yz, yt, zt) is one of MASK_SPATIAL's planes."""
    return MASK_SPATIAL >> (k % 6) & 1


def _product_key(xyz, version, aabb, planes):
    """Identity of everything the spatial product depends on: the same tensors at the same versions.  FusedAdam.step writes
    parameters through raw pointers and bumps their versions explicitly (adam.py), so an optimiser step always changes it."""
    return (xyz.data_ptr(), version, int(xyz.shape[0]), aabb.data_ptr(), aabb._version) + tuple((p.data_ptr(), p._version) for p in planes)


class _SpatialProduct:
    """S[P, 32 levels] = product over the three spatial planes of the bilinear samples at xyz, per level, for the field calls
    whose (xyz, aabb, planes) match `key`.  A trainer step's also holds A, its views' summed dL/dS (A_written: the first view's
    backward has written it), and the xyz leaf and grid of its deferred backward; `auto`: each view's dL/dS goes to autograd."""

    def __init__(self, key, xyz, aabb, planes, levels, res, order, auto=False):
        self.key, self.order, self.auto = key, order, auto
        self.A, self.A_written, self.xyz_param, self.grid = None, False, None, None
        P = int(xyz.shape[0])
        self.S = torch.empty((P, 32 * levels), dtype=torch.float32, device=xyz.device)
        d = _hex_desc(aabb, planes, levels, res)
        check(_lib.lib().b200gs_hexplane_forward_masked(ctypes.byref(d), P, xyz.data_ptr(), _lib.ptr(order), None, 0.0, MASK_SPATIAL, None,
                                                        self.S.data_ptr(), current_stream()), "hexplane_forward(spatial)")
        _lib.COUNTERS["spatial_product_evaluations"] += 1

    def matches(self, xyz, aabb, planes):
        return self.key == _product_key(xyz, xyz._version, aabb, planes)

    @staticmethod
    def backward(dS, xyz, order, aabb, planes, levels, res, grads):
        """dS into `grads` (the spatial planes' gradient buffers, None for the others); returns d_xyz.  Static: _SpatialFn's
        node must not hold the product, which holds that node's output S (a reference cycle)."""
        d = _hex_desc(aabb, planes, levels, res, grads)
        d_xyz = torch.empty_like(xyz)
        check(_lib.lib().b200gs_hexplane_backward_masked(ctypes.byref(d), int(xyz.shape[0]), xyz.data_ptr(), _lib.ptr(order), None, 0.0,
                                                         MASK_SPATIAL, None, None, dS.data_ptr(), d_xyz.data_ptr(), None, 0,
                                                         current_stream()), "hexplane_backward(spatial)")
        return d_xyz

    def view_gradient(self, accumulate_only):
        """Where a view's backward puts its dL/dS: (buffer, whether the kernel writes it rather than adds to it).  Autograd
        holder: a fresh buffer per view, handed back to autograd.  Trainer step: A, written by the step's first view and added
        to by the rest.  A kernel that can only accumulate (accumulate_only) gets the buffer zeroed instead of written."""
        if self.auto:
            buf, first = torch.empty_like(self.S), True
        else:
            buf, first, self.A_written = self.A, not self.A_written, True
        if first and accumulate_only:
            buf.zero_()
        return buf, first and not accumulate_only


_SHARED = None


def begin_shared_step(net, xyz_param, inference=False):
    """net: deform_network; xyz_param: the leaf the views will query (its .grad receives the spatial xyz gradient).
    inference: no gradient accumulator is allocated (see shared_spatial_product)."""
    global _SHARED
    grid = net.deformation_net.grid
    planes = grid._planes()
    xyz = xyz_param.detach().contiguous()
    _check_cuda_f32(xyz, grid.aabb, *planes)
    sh = _SpatialProduct(_product_key(xyz, xyz_param._version, grid.aabb, planes), xyz, grid.aabb, planes, len(grid.grids),
                         tuple(grid._res), _cell_order(xyz, grid.aabb))
    sh.A, sh.xyz_param, sh.grid = None if inference else torch.empty_like(sh.S), xyz_param, grid
    _SHARED = sh


@contextlib.contextmanager
def shared_spatial_product(net, xyz_param):
    """Rendering a sequence of frames of ONE static model (render_4DGS.py:41-76 renders a whole trajectory from fixed
    Gaussians): the product of the three spatial planes depends on xyz only, so it is evaluated once for the sequence and
    every frame samples just its time planes (b200gs_hexplane_time_forward: 1-D lerps from shared memory) and multiplies.
    Same values as the per-frame six-plane pass up to FP32 re-association (tests/test_hexplane_split_parity.py).  Use under
    torch.no_grad(); nothing is accumulated and no backward is deferred.  The model must not change inside the block."""
    global _SHARED
    begin_shared_step(net, xyz_param, inference=True)
    try:
        yield
    finally:
        _SHARED = None


def finish_shared_step():
    """The deferred spatial backward: plane gradients into the planes' .grad, xyz gradient into xyz_param.grad."""
    global _SHARED
    sh, _SHARED = _SHARED, None
    if sh is None or not sh.A_written:
        return          # no view's backward contributed
    grid, xyz_param = sh.grid, sh.xyz_param
    planes = grid._planes()
    grads = [p.grad if _is_spatial(k) else None for k, p in enumerate(planes)]
    if any(_is_spatial(k) and (p.grad is None or p.grad.stride() != p.stride()) for k, p in enumerate(planes)):
        raise RuntimeError("finish_shared_step needs channels-last .grad buffers on the spatial planes")
    xyz = xyz_param.detach().contiguous()
    d_xyz = _SpatialProduct.backward(sh.A, xyz, sh.order, grid.aabb, planes, len(grid.grids), tuple(grid._res), grads)
    if xyz_param.grad is None:
        xyz_param.grad = d_xyz
    else:
        xyz_param.grad += d_xyz


def drop_shared():
    """Forget the per-step / per-sequence spatial product (called by FusedAdam.step and by the trainer's error path)."""
    global _SHARED, _INFER, _AUTO
    _SHARED = None
    _INFER = None
    _AUTO = None


# Opt-in (B200GS_INFERENCE_SPATIAL_CACHE=1 or field.INFERENCE_SPATIAL_CACHE = True; not yet run on a GPU): what
# shared_spatial_product does for a caller that can wrap its frame loop, done implicitly for callers that cannot -- the
# reference's own render_4DGS.py running unchanged through the launcher.  Under torch.no_grad() the spatial product is kept
# between calls for as long as xyz, the aabb and every plane are the same tensors at the same version; FusedAdam.step() writes
# parameters through raw pointers, so it drops the cache explicitly as well.
INFERENCE_SPATIAL_CACHE = os.environ.get("B200GS_INFERENCE_SPATIAL_CACHE") == "1"
_INFER = None


def invalidate_inference_cache():
    global _INFER
    _INFER = None


# ---- the same split under plain autograd (the reference's own training loop through the launcher) ---------------------------
# train_4DGS.py:172-229 renders the views of a batch one after the other and calls loss.backward() ONCE.  The product of the
# three spatial planes is an ordinary differentiable tensor S = _SpatialFn(xyz, planes): it is evaluated once per set of
# parameter versions, every view's field call takes it as an input (time planes from shared memory, hexplane_time_*), autograd
# sums the views' dL/dS and runs the spatial backward once.  The cached S dies with the backward pass that consumes it.
AUTOGRAD_SPATIAL_SHARING = os.environ.get("B200GS_AUTOGRAD_SPATIAL_SHARING", "1") != "0"
_AUTO = None


def _drop_auto(*_):
    global _AUTO
    _AUTO = None


class _SpatialFn(torch.autograd.Function):
    """(S, product) = the autograd holder's _SpatialProduct at xyz and its S, differentiable in xyz and the planes."""

    @staticmethod
    def forward(ctx, key, xyz, aabb, levels, res, *planes):
        xyz = xyz.contiguous()
        _check_cuda_f32(xyz, aabb, *planes)
        product = _SpatialProduct(key, xyz, aabb, planes, levels, res, _cell_order(xyz, aabb), auto=True)
        ctx.save_for_backward(xyz, aabb, *planes)
        ctx.meta = (levels, res)
        ctx.order = product.order
        ctx.params = planes
        return product.S, product

    @staticmethod
    def backward(ctx, dS, _):
        xyz, aabb, *planes = ctx.saved_tensors
        levels, res = ctx.meta
        dS = dS.contiguous()
        direct = [_grad_target(q) if _is_spatial(k) else None for k, q in enumerate(ctx.params)]
        grads = [(dp if dp is not None else torch.zeros_like(p, memory_format=torch.preserve_format)) if _is_spatial(k) else None
                 for k, (p, dp) in enumerate(zip(planes, direct))]
        d_xyz = _SpatialProduct.backward(dS, xyz, ctx.order, aabb, planes, levels, res, grads)
        return (None, d_xyz, None, None, None, *[None if dp is not None else g for g, dp in zip(grads, direct)])


def _auto_spatial(xyz, grid):
    """The differentiable spatial product for this (xyz, planes, aabb) state: cached until a backward pass consumes it or any
    of those tensors changes."""
    global _AUTO
    planes = grid._planes()
    if _AUTO is None or not _AUTO.matches(xyz, grid.aabb, planes):
        S, _AUTO = _SpatialFn.apply(_product_key(xyz, xyz._version, grid.aabb, planes), xyz, grid.aabb, len(grid.grids),
                                    tuple(grid._res), *planes)
        if S.requires_grad:
            S.register_hook(_drop_auto)          # its gradient is being produced: the graph below it is about to be freed
    return _AUTO.S


def _product_for(xyz, aabb, planes, levels, res, order, S_in):
    """The spatial product a field call multiplies its time planes by, or None (all six planes sampled): the explicit scope's
    if it matches, else the autograd holder's if the caller passed its S (S_in, from _auto_spatial), else the implicit no-grad
    cache's (evaluated here on a miss)."""
    global _INFER
    if _SHARED is not None and _SHARED.matches(xyz, aabb, planes):
        return _SHARED
    if S_in is not None:
        return _AUTO
    if not INFERENCE_SPATIAL_CACHE or torch.is_grad_enabled():
        return None
    if _INFER is None or not _INFER.matches(xyz, aabb, planes):
        _INFER = _SpatialProduct(_product_key(xyz, xyz._version, aabb, planes), xyz, aabb, planes, levels, res, order)
    return _INFER


class _DeformFn(torch.autograd.Function):
    """(pts, scales, rot[, opacity'][, shs']) = field(xyz, scales, rot, opacity, shs, t, scene_flow, frame_num, delta_scale).

    inputs: xyz, scales, rot, opacity, shs, times, scene_flow, frame_num, delta_scale, aabb, levels, res, heads, S_in,
            need_backward, w1, b1, (w2,b2,w3,b3) x 5 heads, *planes
    heads: (pos, scales, rotations, opacity, shs) on / off.  opacity' / shs' are returned only for the heads that are on
    (csrc/deform_heads.cu); opacity / shs may be None when their head is off.
    S_in: None, or the autograd holder's differentiable spatial product (_auto_spatial; then only the time planes are sampled
    here and dL/dS_in is returned for autograd to sum over the views of a batch).
    """
    N_FIXED = 15
    N_W = 22

    @staticmethod
    def forward(ctx, xyz, scales, rot, opacity, shs, times, scene_flow, frame_num, delta_scale, aabb, levels, res, heads, S_in,
                need_backward, *rest):
        weights, planes = rest[:_DeformFn.N_W], rest[_DeformFn.N_W:]
        xyz = xyz.contiguous(); scales = scales.contiguous(); rot = rot.contiguous(); scene_flow = scene_flow.contiguous()
        _check_cuda_f32(xyz, scales, rot, scene_flow, aabb, *planes, *[w for w in weights if w is not None])
        L = _lib.lib()
        P = int(xyz.shape[0])
        dev = xyz.device
        stream = current_stream()
        tt, ts = _times_arg(times, P, detect=False)          # (the caller has already looked for a uniform tensor)
        feat = torch.empty((P, 32 * levels), dtype=torch.float32, device=dev)
        d = _hex_desc(aabb, planes, levels, res)
        order = _cell_order(xyz, aabb)
        ctx.order = order
        sh = ctx.product = _product_for(xyz, aabb, planes, levels, res, order, S_in)
        ctx.time_rows = False
        ctx.feat_tiled = False
        if sh is not None and tt is None and L.b200gs_hexplane_time_supported(ctypes.byref(d)):
            # shared spatial product + one timestamp for the view: time planes served from shared memory
            ctx.time_rows = True
            # (no cell order here: with the rows in shared memory there is no texel locality to gain, and walking the points in
            #  storage order keeps the S / feature rows streaming)
            # feature / d_feature rows in the stash's 4-point-group tiles: coalesced for the MLP kernels' lane-per-point access
            ctx.feat_tiled = levels == 2
            if ctx.feat_tiled:
                feat = torch.empty(((P + 127) // 128 * 128, 32 * levels), dtype=torch.float32, device=dev)
            check(L.b200gs_hexplane_time_forward(ctypes.byref(d), P, xyz.data_ptr(), None, ts, sh.S.data_ptr(),
                                                 feat.data_ptr(), int(ctx.feat_tiled), stream), "hexplane_time_forward")
            _lib.COUNTERS["time_row_forward_calls"] += 1
        elif sh is not None:      # shared spatial product, per-point times: only the time planes are sampled per view
            check(L.b200gs_hexplane_forward_masked(ctypes.byref(d), P, xyz.data_ptr(), _lib.ptr(order),
                                                   tt.data_ptr() if tt is not None else None, ts, MASK_TIME, sh.S.data_ptr(),
                                                   feat.data_ptr(), stream), "hexplane_forward(time)")
        else:
            check(L.b200gs_hexplane_forward(ctypes.byref(d), P, xyz.data_ptr(), _lib.ptr(order),
                                            tt.data_ptr() if tt is not None else None, ts, feat.data_ptr(), stream),
                  "hexplane_forward")
        mw = _DeformFn._weights_struct(weights, heads, 32 * levels)
        mw.feat_tiled = int(ctx.feat_tiled)
        extra = heads[3] or heads[4]
        # inference (the caller knows no backward will follow: torch.no_grad() or nothing requires grad): no activation stash,
        # unless the opacity / SH heads run: they read relu(hidden) from it
        stash = need_backward or not all(heads[:3]) or extra
        saved = torch.empty((L.b200gs_deform_mlp_saved_floats(P),), dtype=torch.float32, device=dev) if stash else None
        pts_o = torch.empty_like(xyz); scales_o = torch.empty_like(scales); rot_o = torch.empty_like(rot)
        if torch.is_tensor(frame_num):
            fn_dev = frame_num.to(device=dev, dtype=torch.float32).reshape(-1)[:1].contiguous()
            fn_val, fn_ptr = 0.0, fn_dev.data_ptr()
        else:
            fn_dev, fn_val, fn_ptr = None, float(frame_num), None
        check(L.b200gs_deform_mlp_forward(ctypes.byref(mw), P, feat.data_ptr(), xyz.data_ptr(), scales.data_ptr(),
                                          rot.data_ptr(), scene_flow.data_ptr(), fn_val, fn_ptr, float(delta_scale),
                                          pts_o.data_ptr(), scales_o.data_ptr(), rot_o.data_ptr(), saved.data_ptr() if saved is not None else None, stream),
              "deform_mlp_forward")
        outs = [pts_o, scales_o, rot_o]
        hsaved = torch.empty(0, device=dev)
        if extra:
            op_in = opacity.contiguous() if heads[3] else None
            sh_in = shs.contiguous() if heads[4] else None
            _check_cuda_f32(op_in, sh_in)
            if need_backward:
                hsaved = torch.empty((L.b200gs_deform_heads_saved_floats(P),), dtype=torch.float32, device=dev)
            op_o = torch.empty_like(op_in) if op_in is not None else None
            sh_o = torch.empty_like(sh_in) if sh_in is not None else None
            hw = _DeformFn._heads_struct(weights, heads, 32 * levels, ctx.feat_tiled)
            check(L.b200gs_deform_heads_forward(ctypes.byref(hw), P, _sh_coeffs(sh_in), saved.data_ptr(), _lib.ptr(op_in),
                                                _lib.ptr(sh_in), _lib.ptr(op_o), _lib.ptr(sh_o),
                                                _lib.ptr(hsaved), stream), "deform_heads_forward")
            _lib.COUNTERS["deform_heads_forward"] += 1
            outs += [o for o in (op_o, sh_o) if o is not None]
        if saved is None:
            saved = torch.empty(0, device=dev)
        ctx.save_for_backward(xyz, tt if tt is not None else torch.empty(0), aabb, feat, saved, hsaved,
                              *[w if w is not None else torch.empty(0) for w in weights], *planes)
        ctx.meta = (levels, res, heads, ts, tt is not None)
        ctx.params = (weights, planes)          # the Parameter objects themselves (for _grad_target)
        return tuple(outs)

    @staticmethod
    def _heads_struct(weights, heads, feat_dim, feat_tiled):
        hw = _HeadsWeights()
        hw.feat_dim = feat_dim
        hw.width = int(weights[0].shape[0])
        hw.w1 = weights[0].data_ptr()
        hw.feat_tiled = int(feat_tiled)
        for h in range(2):
            if heads[3 + h]:
                w2, b2, w3, b3 = weights[14 + 4 * h: 18 + 4 * h]
                hw.w2[h], hw.b2[h], hw.w3[h], hw.b3[h] = w2.data_ptr(), b2.data_ptr(), w3.data_ptr(), b3.data_ptr()
        return hw

    @staticmethod
    def _weights_struct(weights, heads, feat_dim):
        mw = _MlpWeights()
        mw.feat_dim = feat_dim
        mw.width = int(weights[0].shape[0])
        mw.w1 = weights[0].data_ptr(); mw.b1 = weights[1].data_ptr()
        for h in range(3):
            w2, b2, w3, b3 = weights[2 + 4 * h: 6 + 4 * h]
            on = heads[h] and w2 is not None and w2.numel() > 0
            mw.w2[h] = w2.data_ptr() if on else None
            mw.b2[h] = b2.data_ptr() if on else None
            mw.w3[h] = w3.data_ptr() if on else None
            mw.b3[h] = b3.data_ptr() if on else None
        return mw

    @staticmethod
    def backward(ctx, d_pts, d_scales, d_rot, *d_extra):
        xyz, tt, aabb, feat, saved, hsaved, *rest = ctx.saved_tensors
        weights, planes = rest[:_DeformFn.N_W], rest[_DeformFn.N_W:]
        levels, res, heads, ts, has_t = ctx.meta
        if saved.numel() == 0:
            raise RuntimeError("deform_network: backward through a forward that ran in inference mode (no activation stash)")
        L = _lib.lib()
        P = int(xyz.shape[0])
        stream = current_stream()
        mw = _DeformFn._weights_struct(weights, heads, 32 * levels)
        mw.feat_tiled = int(ctx.feat_tiled)
        pw, pp = ctx.params
        direct_w = [_grad_target(q) if q is not None else None for q in pw]
        direct_p = [_grad_target(q) for q in pp]
        # (the weights of a disabled opacity / SH head get no buffer: with both off nothing is allocated beyond the three heads)
        live = [i < 14 or heads[3 + (i - 14) // 4] for i in range(len(weights))]
        gws = [(dw if dw is not None else torch.zeros_like(w)) if (w.numel() and on) else None
               for w, dw, on in zip(weights, direct_w, live)]
        mg = _MlpGrads()
        mg.w1 = gws[0].data_ptr(); mg.b1 = gws[1].data_ptr()
        for h in range(3):
            for name, i in (("w2", 2), ("b2", 3), ("w3", 4), ("b3", 5)):
                g = gws[i + 4 * h]
                getattr(mg, name)[h] = g.data_ptr() if (g is not None and heads[h]) else None
        d_feat = torch.empty_like(feat)
        # contiguous copies of the upstream gradients stay referenced until the launch has been queued
        d_pts, d_scales, d_rot = (t.contiguous() if t is not None else None for t in (d_pts, d_scales, d_rot))
        check(L.b200gs_deform_mlp_backward(ctypes.byref(mw), ctypes.byref(mg), P, feat.data_ptr(), saved.data_ptr(),
                                           _lib.ptr(d_pts) if heads[0] else None, _lib.ptr(d_scales) if heads[1] else None,
                                           _lib.ptr(d_rot) if heads[2] else None, d_feat.data_ptr(), stream), "deform_mlp_backward")
        d_op = d_sh = None
        if heads[3] or heads[4]:
            if hsaved.numel() == 0:
                raise RuntimeError("deform_network: backward through a forward that ran in inference mode (no heads stash)")
            # after the three-head backward (which WROTE d_feat, dW1, db1) and before the HexPlane backward reads d_feat
            d_extra = [t.contiguous() if t is not None else None for t in d_extra]
            d_op = d_extra[0] if heads[3] else None
            d_sh = d_extra[-1] if heads[4] else None
            acc = SH_GRAD_ACCUMULATOR
            use_acc = (d_sh is not None and acc is not None and acc.shape == d_sh.shape and acc.is_contiguous()
                       and acc.device == d_sh.device and acc.dtype == torch.float32)
            hg = _HeadsGrads()
            hg.w1 = gws[0].data_ptr(); hg.b1 = gws[1].data_ptr()
            for h in range(2):
                if heads[3 + h]:
                    hg.w2[h], hg.b2[h], hg.w3[h], hg.b3[h] = (gws[i].data_ptr() for i in range(14 + 4 * h, 18 + 4 * h))
            hw = _DeformFn._heads_struct(weights, heads, 32 * levels, ctx.feat_tiled)
            check(L.b200gs_deform_heads_backward(ctypes.byref(hw), ctypes.byref(hg), P, _sh_coeffs(d_sh), feat.data_ptr(),
                                                 saved.data_ptr(), hsaved.data_ptr(), _lib.ptr(d_op), _lib.ptr(d_sh), d_feat.data_ptr(),
                                                 acc.data_ptr() if use_acc else None, int(use_acc and SH_GRAD_OVERWRITE), stream),
                  "deform_heads_backward")
            _lib.COUNTERS["deform_heads_backward"] += 1
            if use_acc:
                d_sh = None                     # already in the step's SH buffer
        if AFTER_MLP_BACKWARD is not None:
            AFTER_MLP_BACKWARD()
        sh = ctx.product
        # the spatial planes receive nothing here when only the time planes were sampled (their share goes through S)
        gplanes = [dp if dp is not None else (None if (sh is not None and _is_spatial(k)) else torch.zeros_like(p, memory_format=torch.preserve_format))
                   for k, (p, dp) in enumerate(zip(planes, direct_p))]
        d_xyz_grid = torch.empty_like(xyz)
        d = _hex_desc(aabb, planes, levels, res, gplanes)
        dS = None
        if ctx.time_rows:
            scratch, nbytes = _time_row_scratch(d, xyz.device)
            dS, overwrite = sh.view_gradient(accumulate_only=False)
            check(L.b200gs_hexplane_time_backward(ctypes.byref(d), P, xyz.data_ptr(), None, ts, sh.S.data_ptr(),
                                                  dS.data_ptr(), d_feat.data_ptr(), d_xyz_grid.data_ptr(), scratch.data_ptr(),
                                                  nbytes, int(ctx.feat_tiled) | (2 if overwrite else 0), stream), "hexplane_time_backward")
        elif sh is not None or not has_t:
            # shared product: time planes now, the spatial planes' share goes into this view's dL/dS.
            # One timestamp for the whole launch (scalar time): the time planes' gradient goes through replicated 1-D rows.
            scratch, nbytes = _time_row_scratch(d, xyz.device) if not has_t else (None, 0)
            if sh is not None:
                dS, _ = sh.view_gradient(accumulate_only=True)
            check(L.b200gs_hexplane_backward_masked(ctypes.byref(d), P, xyz.data_ptr(), _lib.ptr(ctx.order),
                                                    tt.data_ptr() if has_t else None, ts, MASK_TIME if sh is not None else MASK_ALL,
                                                    sh.S.data_ptr() if sh is not None else None, _lib.ptr(dS), d_feat.data_ptr(),
                                                    d_xyz_grid.data_ptr(), _lib.ptr(scratch), nbytes, stream), "hexplane_backward(time)")
        else:
            check(L.b200gs_hexplane_backward(ctypes.byref(d), P, xyz.data_ptr(), _lib.ptr(ctx.order),
                                             tt.data_ptr() if has_t else None, ts, d_feat.data_ptr(), d_xyz_grid.data_ptr(),
                                             stream), "hexplane_backward")
        d_S = dS if sh is not None and sh.auto else None        # the autograd holder's views: autograd sums dL/dS
        # pts = xyz*1 + ..., scales = scales*1 + ds, rot = rot + dr: identity paths
        d_xyz = d_xyz_grid + d_pts if d_pts is not None else d_xyz_grid
        gw_out = [None if dw is not None else g for g, dw in zip(gws, direct_w)]      # accumulated in place -> nothing for autograd
        for h in range(5):
            if not heads[h]:
                for i in range(2 + 4 * h, 6 + 4 * h):
                    gw_out[i] = None
        gp_out = [None if dp is not None else g for g, dp in zip(gplanes, direct_p)]
        # opacity' = opacity * 1 + ..., shs' = shs * 1 + ...: identity paths
        return (d_xyz, d_scales, d_rot, d_op, d_sh, None, None, None, None, None, None, None, None, d_S, None, *gw_out, *gp_out)


def _sh_coeffs(shs):
    """SH coefficients per point of a [P, M, 3] tensor (None: no SH head), -1 for any other shape (the kernels refuse it)."""
    if shs is None:
        return 16
    return int(shs.shape[1]) if shs.dim() == 3 and shs.shape[2] == 3 else -1


def _regulation_launch(field, weights, loss_accum, grads):
    planes = field._planes()
    levels = len(field.grids)
    d = _hex_desc(field.aabb, planes, levels, tuple(field._res), grads)
    tw, l1w, pw = weights
    check(_lib.lib().b200gs_hexplane_regulation(ctypes.byref(d), float(pw), float(tw), float(l1w),
                                                loss_accum.data_ptr() if loss_accum is not None else None, current_stream()),
          "hexplane_regulation")


class _RegulationFn(torch.autograd.Function):
    """compute_regulation (scene/gaussian_model.py:768-769) as one kernel each way."""

    @staticmethod
    def forward(ctx, field, tw, l1w, pw, *planes):
        loss = torch.zeros(1, dtype=torch.float32, device=planes[0].device)
        _regulation_launch(field, (tw, l1w, pw), loss, None)
        ctx.field, ctx.weights = field, (tw, l1w, pw)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, g):
        planes = ctx.field._planes()
        grads = [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes]
        _regulation_launch(ctx.field, ctx.weights, None, grads)
        return (None, None, None, None, *[gr * g for gr in grads])


def compute_regulation(field, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight):
    """Drop-in for GaussianModel.compute_regulation (scene/gaussian_model.py:768-769; same argument order) given the
    HexPlaneField: differentiable scalar."""
    return _RegulationFn.apply(field, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight, *field._planes())


def accumulate_regulation(field, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight, loss_accum=None):
    """Trainer fast path: add the regulariser's gradient straight into the planes' existing `.grad` buffers (and its value
    into `loss_accum`), one launch, no autograd."""
    grads = []
    for p in field._planes():
        if p.grad is None or p.grad.stride() != p.stride():
            raise RuntimeError("accumulate_regulation needs channels-last .grad buffers on every plane")
        grads.append(p.grad)
    _regulation_launch(field, (time_smoothness_weight, l1_time_planes_weight, plane_tv_weight), loss_accum, grads)


# ---------------------------------------------------------------------------------------------
# modules (same structure as the reference so state_dicts and the optimiser groups line up)
# ---------------------------------------------------------------------------------------------
def init_grid_param(grid_nd, in_dim, out_dim, reso, a=0.1, b=0.5):
    """scene/hexplane.py:48-70; returns channels_last parameters."""
    assert in_dim == len(reso), "Resolution must have same number of elements as input-dimension"
    has_time_planes = in_dim == 4
    assert grid_nd <= in_dim
    grid_coefs = nn.ParameterList()
    for coo_comb in itertools.combinations(range(in_dim), grid_nd):
        t = torch.empty([1, out_dim] + [reso[cc] for cc in coo_comb[::-1]])
        if has_time_planes and 3 in coo_comb:
            nn.init.ones_(t)
        else:
            nn.init.uniform_(t, a=a, b=b)
        grid_coefs.append(nn.Parameter(_cl(t)))
    return grid_coefs


class HexPlaneField(nn.Module):
    def __init__(self, bounds, planeconfig, multires) -> None:
        super().__init__()
        aabb = torch.tensor([[bounds, bounds, bounds], [-bounds, -bounds, -bounds]])
        self.aabb = nn.Parameter(aabb, requires_grad=False)
        self.grid_config = [planeconfig]
        self.multiscale_res_multipliers = multires
        self.concat_features = True
        cfg0 = self.grid_config[0]
        if not HexPlaneField.supports(planeconfig, multires):
            raise NotImplementedError("b200gs HexPlaneField supports 2-D planes over (x, y, z, t) with 16 or 32 channels at "
                                      f"1-{MAX_LEVELS} levels (got {cfg0['grid_dimensions']}-D over {cfg0['input_coordinate_dim']} "
                                      f"coordinates, {cfg0['output_coordinate_dim']} channels, {len(multires)} levels)")
        self.grids = nn.ModuleList()
        self.feat_dim = 0
        self._res = []
        for res in self.multiscale_res_multipliers:
            config = cfg0.copy()
            config["resolution"] = [r * res for r in config["resolution"][:3]] + config["resolution"][3:]
            gp = init_grid_param(grid_nd=config["grid_dimensions"], in_dim=config["input_coordinate_dim"],
                                 out_dim=config["output_coordinate_dim"], reso=config["resolution"])
            self.feat_dim += gp[-1].shape[1]
            self.grids.append(gp)
            self._res.append(tuple(int(r) for r in config["resolution"]))
        print("feature_dim:", self.feat_dim)

    @staticmethod
    def supports(planeconfig, multires):
        """Whether the kernels cover this (kplanes_config, multires): 2-D planes over (x, y, z, t), 16 or 32 channels,
        1-4 levels."""
        return (planeconfig["grid_dimensions"] == 2 and planeconfig["input_coordinate_dim"] == 4
                and planeconfig["output_coordinate_dim"] in (16, 32) and 1 <= len(multires) <= MAX_LEVELS)

    @property
    def get_aabb(self):
        return self.aabb[0], self.aabb[1]

    def set_aabb(self, xyz_max, xyz_min):
        aabb = torch.tensor([xyz_max, xyz_min], dtype=torch.float32)
        self.aabb = nn.Parameter(aabb.to(self.aabb.device), requires_grad=False)
        print("Voxel Plane: set aabb=", self.aabb)

    def _planes(self):
        out = []
        for gp in self.grids:
            for p in gp:
                if p.stride(1) != 1:           # e.g. after load_state_dict into a re-created parameter
                    p.data = _cl(p.data)
                out.append(p)
        return out

    def _time_rows_supported(self):
        """Can the one-timestamp kernels (time planes pre-blended in shared memory) serve this configuration?"""
        if self.aabb.is_cuda:
            d = _hex_desc(self.aabb, self._planes(), len(self.grids), tuple(self._res))
            return bool(_lib.lib().b200gs_hexplane_time_supported(ctypes.byref(d)))
        return False

    def get_density(self, pts, timestamps=None):
        if timestamps is None:
            raise NotImplementedError("static (time-free) HexPlane queries are not on the reference's path")
        pts = pts.reshape(-1, pts.shape[-1])
        return _HexPlaneFn.apply(pts[:, :3], timestamps, self.aabb, len(self.grids), tuple(self._res), *self._planes())

    def forward(self, pts, timestamps=None):
        return self.get_density(pts, timestamps)


def _head(W, k):
    return nn.Sequential(nn.ReLU(), nn.Linear(W, W), nn.ReLU(), nn.Linear(W, k))


class Deformation(nn.Module):
    def __init__(self, D=8, W=256, input_ch=27, input_ch_time=9, grid_pe=0, skips=[], args=None):
        super().__init__()
        self.D = D
        self.W = W
        self.input_ch = input_ch
        self.input_ch_time = input_ch_time
        self.skips = skips
        self.grid_pe = grid_pe
        self.no_grid = args.no_grid
        # the MLP kernels take a 64- or 128-wide feature row: 32 channels at 2 or 4 levels (checked before the grid consumes
        # any random numbers)
        if args.kplanes_config["output_coordinate_dim"] != 32 or len(args.multires) not in (2, 4):
            raise NotImplementedError("b200gs Deformation: the fused MLP needs 32 channels per plane at 2 or 4 levels (got "
                                      f"{args.kplanes_config['output_coordinate_dim']} channels, {len(args.multires)} levels)")
        self.grid = HexPlaneField(args.bounds, args.kplanes_config, args.multires)
        self.args = args
        unsupported = []
        if args.no_grid: unsupported.append("no_grid")
        if args.empty_voxel: unsupported.append("empty_voxel")
        if args.static_mlp: unsupported.append("static_mlp")
        if grid_pe != 0: unsupported.append("grid_pe")
        if getattr(args, "apply_rotation", False): unsupported.append("apply_rotation")
        if D > 1: unsupported.append("defor_depth>1")
        if W != 64: unsupported.append("net_width!=64")
        if unsupported:
            raise NotImplementedError("b200gs Deformation: configuration outside the fused kernels' scope: " + ", ".join(unsupported))
        self.ratio = 0
        self.create_net()

    @property
    def get_aabb(self):
        return self.grid.get_aabb

    def set_aabb(self, xyz_max, xyz_min):
        print("Deformation Net Set aabb", xyz_max, xyz_min)
        self.grid.set_aabb(xyz_max, xyz_min)

    def create_net(self):
        feature_out = [nn.Linear(self.grid.feat_dim, self.W)]
        for _ in range(self.D - 1):
            feature_out.append(nn.ReLU())
            feature_out.append(nn.Linear(self.W, self.W))
        self.feature_out = nn.Sequential(*feature_out)
        self.pos_deform = _head(self.W, 3)
        self.scales_deform = _head(self.W, 3)
        self.rotations_deform = _head(self.W, 4)
        self.opacity_deform = _head(self.W, 1)
        self.shs_deform = _head(self.W, 16 * 3)

    @property
    def get_empty_ratio(self):
        return self.ratio

    def forward(self, rays_pts_emb, scales_emb=None, rotations_emb=None, opacity=None, shs_emb=None, time_feature=None,
                time_emb=None, scene_flow=None, frame_num=None, delta_scale=None):
        if time_emb is None:
            raise NotImplementedError("forward_static needs static_mlp, which the reference does not enable")
        return self.forward_dynamic(rays_pts_emb, scales_emb, rotations_emb, opacity, shs_emb, time_feature, time_emb,
                                    scene_flow, frame_num, delta_scale)

    def forward_dynamic(self, rays_pts_emb, scales_emb, rotations_emb, opacity_emb, shs_emb, time_feature, time_emb,
                        scene_flow, frame_num, delta_scale):
        a = self.args
        heads = (not a.no_dx, not a.no_ds, not a.no_dr, not a.no_do, not a.no_dshs)
        weights = [self.feature_out[0].weight, self.feature_out[0].bias]
        for m in (self.pos_deform, self.scales_deform, self.rotations_deform, self.opacity_deform, self.shs_deform):
            weights += [m[1].weight, m[1].bias, m[3].weight, m[3].bias]
        xyz = rays_pts_emb[:, :3]
        if scene_flow is None:
            scene_flow = torch.zeros_like(xyz)
        if frame_num is None:
            frame_num = 0.0
        if delta_scale is None:
            delta_scale = 0.0
        # time_emb: the reference's [P,1] tensor (gaussian_renderer/__init__.py:56), or one Python float for the whole call
        t_arg = time_emb[:, :1] if torch.is_tensor(time_emb) else float(time_emb)
        S_in = None
        need_backward = torch.is_grad_enabled() and (any(t.requires_grad for t in (rays_pts_emb, scales_emb, rotations_emb))
                                                     or (heads[3] and opacity_emb.requires_grad) or (heads[4] and shs_emb.requires_grad)
                                                     or any(w.requires_grad for w in weights) or self.grid.grids[0][0].requires_grad)
        if torch.is_tensor(t_arg) and xyz.is_cuda:
            # the reference's render() hands over the camera's ONE timestamp as a [P,1] tensor (gaussian_renderer/__init__.py:56)
            tt, ts = _times_arg(t_arg, int(xyz.shape[0]))
            t_arg = ts if tt is None else tt
        if (AUTOGRAD_SPATIAL_SHARING and not torch.is_tensor(t_arg) and xyz.is_cuda and torch.is_grad_enabled() and _SHARED is None
                and self.grid._time_rows_supported() and (xyz.requires_grad or self.grid.grids[0][0].requires_grad)):
            S_in = _auto_spatial(xyz, self.grid)
        if heads[4] and not (shs_emb.dim() == 3 and tuple(shs_emb.shape[1:]) == (16, 3)):
            raise NotImplementedError(f"b200gs Deformation: the SH head needs shs of shape [P,16,3], got {tuple(shs_emb.shape)}")
        out = _DeformFn.apply(xyz, scales_emb[:, :3], rotations_emb[:, :4], opacity_emb[:, :1] if heads[3] else None,
                              shs_emb if heads[4] else None, t_arg, scene_flow, frame_num, delta_scale, self.grid.aabb,
                              len(self.grid.grids), tuple(self.grid._res), heads, S_in, need_backward, *weights,
                              *self.grid._planes())
        pts, scales, rotations = out[:3]
        opacity = out[3] if heads[3] else opacity_emb[:, :1]
        shs = out[-1] if heads[4] else shs_emb
        return pts, scales, rotations, opacity, shs

    def get_mlp_parameters(self):
        return [p for n, p in self.named_parameters() if "grid" not in n]

    def get_grid_parameters(self):
        return [p for n, p in self.named_parameters() if "grid" in n]


class deform_network(nn.Module):
    def __init__(self, args):
        super().__init__()
        net_width = args.net_width
        timebase_pe = args.timebase_pe
        defor_depth = args.defor_depth
        posbase_pe = args.posebase_pe
        scale_rotation_pe = args.scale_rotation_pe
        opacity_pe = args.opacity_pe
        timenet_width = args.timenet_width
        timenet_output = args.timenet_output
        grid_pe = args.grid_pe
        times_ch = 2 * timebase_pe + 1
        self.timenet = nn.Sequential(nn.Linear(times_ch, timenet_width), nn.ReLU(), nn.Linear(timenet_width, timenet_output))
        self.deformation_net = Deformation(W=net_width, D=defor_depth, input_ch=(3) + (3 * (posbase_pe)) * 2,
                                           grid_pe=grid_pe, input_ch_time=timenet_output, args=args)
        self.register_buffer('time_poc', torch.FloatTensor([(2 ** i) for i in range(timebase_pe)]))
        self.register_buffer('pos_poc', torch.FloatTensor([(2 ** i) for i in range(posbase_pe)]))
        self.register_buffer('rotation_scaling_poc', torch.FloatTensor([(2 ** i) for i in range(scale_rotation_pe)]))
        self.register_buffer('opacity_poc', torch.FloatTensor([(2 ** i) for i in range(opacity_pe)]))
        self.apply(initialize_weights)

    def forward(self, point, scales=None, rotations=None, opacity=None, shs=None, times_sel=None, scene_flow=None,
                frame_num=None, delta_scale=None):
        return self.forward_dynamic(point, scales, rotations, opacity, shs, times_sel, scene_flow, frame_num, delta_scale)

    @property
    def get_aabb(self):
        return self.deformation_net.get_aabb

    @property
    def get_empty_ratio(self):
        return self.deformation_net.get_empty_ratio

    def forward_dynamic(self, point, scales=None, rotations=None, opacity=None, shs=None, times_sel=None, scene_flow=None,
                        frame_num=None, delta_scale=None):
        # the reference embeds point/scales/rotations with sin/cos here and then uses only the raw
        # leading columns (deformation.py:205-207, :107-135); the raw tensors are passed directly
        return self.deformation_net(point, scales, rotations, opacity, shs, None, times_sel, scene_flow, frame_num,
                                    delta_scale)

    def get_mlp_parameters(self):
        return self.deformation_net.get_mlp_parameters() + list(self.timenet.parameters())

    def get_grid_parameters(self):
        return self.deformation_net.get_grid_parameters()


def initialize_weights(m):
    # scene/deformation.py:229-235 (xavier twice when a bias exists; same RNG consumption)
    if isinstance(m, nn.Linear):
        init.xavier_uniform_(m.weight, gain=1)
        if m.bias is not None:
            init.xavier_uniform_(m.weight, gain=1)


def poc_fre(input_data, poc_buf):
    input_data_emb = (input_data.unsqueeze(-1) * poc_buf).flatten(-2)
    return torch.cat([input_data, input_data_emb.sin(), input_data_emb.cos()], -1)
