"""Run the reference's own scripts, byte-identical, on top of the B200 kernels.

    python -m b200gs.launcher --reference /path/to/ICLR2025_3D-MOM train_4DGS.py -s <scene> --expname <name> ...
    python -m b200gs.launcher --reference /path/to/ICLR2025_3D-MOM render_4DGS.py --input_dir <dir> ...

`install()` (1) puts the drop-in `diff_gaussian_rasterization` / `simple_knn` packages in front of the
reference's compiled extensions, (2) appends import shims for third-party modules this image lacks
(compat/, SURVEY.md Appendix E), (3) swaps `deform_network` for the fused-kernel module where
`GaussianModel` looks it up (scene/gaussian_model.py:21,53), (4) makes `training_setup` build the fused
multi-tensor Adam from the very param groups the reference assembles (gaussian_model.py:197-209), and
(5) installs the one-launch prune / cat bookkeeping (gaussian_model.py:424-482), (6) routes
`compute_regulation` (gaussian_model.py:768-769) to the fused plane-regulariser kernel, (7) routes
`utils.loss_utils.ssim` (the opt.lambda_dssim term) to the fused SSIM kernels (patch_loss_utils), and (8) gives the
reference's own `Deformation` -- built for the configurations (3) leaves to it -- our `HexPlaneField` as its grid
(patch_hexplane), so only its MLP stays in PyTorch. The reference tree is never modified.
"""
import os
import runpy
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_PKG = os.path.dirname(_HERE)


def _library_version_shims():
    """The reference pins torch 1.13 / an old Pillow (README.md:47); two calls it makes are rejected by the versions in this
    image, neither on the GPU path:
      * `torch.load(path)` of its own stage-1 files (PIL images, numpy arrays inside train_data.pth;
        scene/dataset_readers.py:1028) needs the pre-2.6 default weights_only=False;
      * `Image.fromarray(np.array(arr*255.0, dtype=np.byte), "RGB")` (scene/dataset_readers.py:1050; the result is discarded):
        Pillow >= 11 refuses int8 data, older ones reinterpreted it as uint8."""
    os.environ.setdefault("TORCH_FORCE_NO_WEIGHTS_ONLY_LOAD", "1")
    try:
        import numpy as np
        from PIL import Image
    except ImportError:
        return
    if getattr(Image.fromarray, "_b200gs_int8", False):
        return
    real = Image.fromarray

    def fromarray(obj, mode=None, *a, **k):
        if isinstance(obj, np.ndarray) and obj.dtype == np.int8:
            obj = obj.view(np.uint8)
        return real(obj, mode, *a, **k)
    fromarray._b200gs_int8 = True
    Image.fromarray = fromarray


def fused_ssim_supported(img1, img2, window_size=11, size_average=True):
    """Whether fusedops.ssim computes what utils/loss_utils.py:ssim would for these arguments: window 11, two float32 CUDA
    tensors of one shape [N,C,H,W] (or [C,H,W] with size_average, which the reference reduces with .mean() only), no
    gradient wanted for img2.  Looks at metadata only; launches nothing."""
    import torch
    if window_size != 11 or not (isinstance(img1, torch.Tensor) and isinstance(img2, torch.Tensor)):
        return False
    if not (img1.is_cuda and img2.is_cuda and img1.device == img2.device):
        return False
    if img1.dtype != torch.float32 or img2.dtype != torch.float32 or img1.shape != img2.shape or img1.numel() == 0:
        return False
    if not (img1.dim() == 4 or (img1.dim() == 3 and size_average)):
        return False
    return not (img2.requires_grad and torch.is_grad_enabled())


def patch_loss_utils(module):
    """Replaces `module.ssim` (the reference's utils.loss_utils) by a wrapper that sends the calls fusedops.ssim covers
    (fused_ssim_supported) to the fused kernels and every other call to the original function.  Idempotent.
    B200GS_FUSED_SSIM=0 leaves the module as it is.  Returns the module."""
    if os.environ.get("B200GS_FUSED_SSIM", "1") == "0":
        return module
    orig = getattr(module, "ssim", None)
    if orig is None or getattr(orig, "_b200gs_fused", False):
        return module

    def ssim(img1, img2, window_size=11, size_average=True):
        if fused_ssim_supported(img1, img2, window_size, size_average):
            from . import fusedops
            return fusedops.ssim(img1, img2, window_size, size_average)
        return orig(img1, img2, window_size, size_average)
    ssim._b200gs_fused = True
    ssim._b200gs_original = orig
    ssim.__doc__ = orig.__doc__
    module.ssim = ssim
    return module


def patch_hexplane(module):
    """Replaces `module.HexPlaneField` (the name the reference's scene/deformation.py constructs `Deformation.grid` with) by a
    factory that returns b200gs.field.HexPlaneField for the configurations its kernels cover (16 or 32 channels, 1-4 levels,
    2-D planes over x, y, z, t) and the module's original class for any other, with one line on stderr.  Same constructor
    arguments, `feat_dim`, attribute paths and state_dict keys either way.  Idempotent.  Returns the module."""
    orig = getattr(module, "HexPlaneField", None)
    if orig is None or getattr(orig, "_b200gs_factory", False):
        return module
    from . import field

    def HexPlaneField(bounds, planeconfig, multires):
        if field.HexPlaneField.supports(planeconfig, multires):
            return field.HexPlaneField(bounds, planeconfig, multires)
        print(f"[b200gs] HexPlane grid {planeconfig} x {len(multires)} levels is outside the kernels' scope; using the "
              f"reference's {orig.__module__}.HexPlaneField", file=sys.stderr)
        return orig(bounds, planeconfig, multires)
    HexPlaneField._b200gs_factory = True
    HexPlaneField._b200gs_original = orig
    module.HexPlaneField = HexPlaneField
    return module


def install(reference_root):
    reference_root = os.path.abspath(reference_root)
    _library_version_shims()
    for p in (reference_root, _PKG, os.path.join(_PKG, "dropin")):
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    compat = os.path.join(_PKG, "compat")
    if compat not in sys.path:
        sys.path.append(compat)            # last: real installations win
    import scene.gaussian_model as gm       # the reference's module (imports scene.deformation etc.)
    from . import densify, field
    # render_4DGS.py renders whole camera paths from one static model under torch.no_grad(): keep the spatial half of the HexPlane
    # field between frames (dropped as soon as any parameter changes; B200GS_INFERENCE_SPATIAL_CACHE=0 turns it off)
    if os.environ.get("B200GS_INFERENCE_SPATIAL_CACHE") != "0":
        field.INFERENCE_SPATIAL_CACHE = True
    from .adam import FusedAdam
    from .field import deform_network
    reference_deform_network = gm.deform_network

    def make_deform_network(args):
        """scene/gaussian_model.py:53 calls `deform_network(args)`: the fused module for the configurations its kernels cover
        (the one train_4DGS.py trains with by default: width 64, 32 channels, 2 or 4 levels, no_do / no_dshs), the reference's
        own PyTorch module -- on top of the same rasterizer / Adam / densify drop-ins -- for everything else
        (e.g. arguments/dynerf/default.py, arguments/hypernerf/default.py)."""
        try:
            net = deform_network(args)
            _print_summary.field = type(net).__module__
            return net
        except NotImplementedError as ex:
            _print_summary.field = "scene.deformation"
            print(f"[b200gs] {ex}; using the reference's scene.deformation.deform_network for the field", file=sys.stderr)
            return reference_deform_network(args)
    if getattr(reference_deform_network, "__name__", "") != "make_deform_network":
        gm.deform_network = make_deform_network
    # the reference's Deformation (the fallback above) builds its grid from this module's namespace
    import scene.deformation
    patch_hexplane(scene.deformation)
    densify.patch_gaussian_model(gm.GaussianModel)
    if not getattr(gm.GaussianModel, "_b200gs_patched", False):
        for name in ("training_setup", "training_setup_jih"):
            if not hasattr(gm.GaussianModel, name):
                continue
            orig = getattr(gm.GaussianModel, name)

            def wrapped(self, *a, __orig=orig, **k):
                out = __orig(self, *a, **k)
                groups = [{kk: vv for kk, vv in g.items() if kk in ("params", "lr", "name")} for g in self.optimizer.param_groups]
                self.optimizer = FusedAdam(groups, lr=0.0, eps=1e-15)
                _print_summary.optimizer = type(self.optimizer).__name__
                if os.environ.get("B200GS_FUSED_DENSIFY", "1") != "0" and self._xyz.is_cuda:
                    densify.warmup(self)         # first-use kernel loading + allocator growth outside the first densification event
                return out
            setattr(gm.GaussianModel, name, wrapped)
        orig_reg = gm.GaussianModel.compute_regulation

        def compute_regulation(self, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight, __orig=orig_reg):
            from . import field
            grid = self._deformation.deformation_net.grid
            if isinstance(grid, field.HexPlaneField) and grid.aabb.is_cuda:
                return field.compute_regulation(grid, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight)
            return __orig(self, time_smoothness_weight, l1_time_planes_weight, plane_tv_weight)
        gm.GaussianModel.compute_regulation = compute_regulation
        gm.GaussianModel._b200gs_patched = True
    # train_4DGS.py imports `ssim` from utils.loss_utils when it starts (after this point): the lambda_dssim term runs fused
    try:
        import utils.loss_utils as loss_utils
    except ImportError:                     # a script that cannot import it cannot call its ssim either
        loss_utils = None
    if loss_utils is not None:
        patch_loss_utils(loss_utils)
    return gm


def _print_summary(gm):
    from . import _lib
    c = _lib.COUNTERS
    print("[b200gs] launcher summary: field=%s optimizer=%s adam_steps=%d densify_cat_events=%d prune_events=%d raster_forward_calls=%d "
          "time_row_forward_calls=%d spatial_product_evaluations=%d iters_per_s=%.3f"
          % (_print_summary.field, _print_summary.optimizer, c["adam_steps"], c["densify_cat_events"], c["prune_events"],
             c["raster_forward_calls"], c["time_row_forward_calls"], c["spatial_product_evaluations"],
             (c["adam_steps"] - 1) / max(_lib.TIMES.get("last_adam_step", 0.0) - _lib.TIMES.get("first_adam_step", 0.0), 1e-9)
             if c["adam_steps"] > 1 else 0.0), file=sys.stderr, flush=True)


_print_summary.field = "none"
_print_summary.optimizer = "none"


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    if len(argv) < 3 or argv[0] != "--reference":
        raise SystemExit(__doc__)
    ref, script, rest = argv[1], argv[2], argv[3:]
    gm = install(ref)
    if os.environ.get("B200GS_LAUNCHER_LOG") == "1":
        import atexit
        atexit.register(_print_summary, gm)
    path = script if os.path.isabs(script) else os.path.join(os.path.abspath(ref), script)
    os.chdir(os.path.abspath(ref))          # the scripts use paths relative to the repository root
    sys.argv = [path] + rest
    runpy.run_path(path, run_name="__main__")


if __name__ == "__main__":
    main()
