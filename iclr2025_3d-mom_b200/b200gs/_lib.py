"""ctypes binding of libb200gs.so (the C ABI declared in include/b200gs.h).

The product path has no CPU or PyTorch fallback: if the CUDA library is missing or fails
to load, importing anything that needs it raises immediately.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_longlong, c_size_t, c_void_p, POINTER, c_ulonglong

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200gs.so")

_lib = None
# cheap host-side event counts (what ran, how often): read by b200gs.launcher's exit summary and by tests
import collections
COUNTERS = collections.Counter()
TIMES = {}


class B200GSError(RuntimeError):
    """Raised when a libb200gs entry point reports an error (mirrors the RuntimeError the
    reference's pybind layer raises from AT_ERROR / CUDA failures)."""


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `make -C iclr2025_3d-mom_b200/csrc` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        _lib = ctypes.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def _declare(L):
    P = c_void_p
    L.b200gs_last_error.restype = c_char_p
    L.b200gs_last_error.argtypes = []
    L.b200gs_version.restype = c_int
    L.b200gs_set_option.restype = c_int
    L.b200gs_set_option.argtypes = [c_char_p, c_int]
    L.b200gs_get_option.restype = c_int
    L.b200gs_get_option.argtypes = [c_char_p]
    L.b200gs_rast_buffer_sizes.restype = c_int
    L.b200gs_rast_buffer_sizes.argtypes = [c_int, c_longlong, c_int, c_int, POINTER(c_size_t)]
    L.b200gs_rast_forward_stage1.restype = c_int
    L.b200gs_rast_forward_stage1.argtypes = (
        [c_int] * 5 + [P, P, P, P, P, c_float, P, P, P, P, P, c_float, c_float, c_int, P, P, c_size_t, P, P])
    L.b200gs_rast_forward_stage2.restype = c_int
    L.b200gs_rast_forward_stage2.argtypes = [c_int, c_longlong, c_longlong, c_int, c_int, P, P, P, c_size_t, P,
                                             c_size_t, P, P, P]
    L.b200gs_rast_backward.restype = c_int
    L.b200gs_rast_backward.argtypes = (
        [c_int, c_int, c_int, c_longlong, c_int, c_int, P, P, P, P, P, c_float, P, P, P, P, P, c_float, c_float,
         P, P, P, P, P, P, P, P, P, P, P, P, P, P, P, P])
    L.b200gs_rast_backward_accumulate_sh.restype = c_int
    L.b200gs_rast_backward_accumulate_sh.argtypes = L.b200gs_rast_backward.argtypes
    L.b200gs_mark_visible.restype = c_int
    L.b200gs_mark_visible.argtypes = [c_int, P, P, P, P, P]
    L.b200gs_rast_export.restype = c_longlong
    L.b200gs_rast_export.argtypes = [c_char_p, c_int, c_longlong, c_int, c_int, P, P, P, P, c_longlong, P]
    L.b200gs_sort_temp_bytes.restype = c_size_t
    L.b200gs_sort_temp_bytes.argtypes = [c_size_t, c_int, c_int]
    L.b200gs_sort_pairs_u32.restype = c_int
    L.b200gs_sort_pairs_u32.argtypes = [P, P, P, P, c_size_t, c_int, c_int, P, c_size_t, P]
    L.b200gs_dist2_scratch_bytes.restype = c_size_t
    L.b200gs_dist2_scratch_bytes.argtypes = [c_size_t]
    L.b200gs_dist2.restype = c_int
    L.b200gs_dist2.argtypes = [c_int, P, P, P, c_size_t, P]
    for name, (res, args) in _OPTIONAL.items():
        if hasattr(L, name):
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args


# entry points added by later translation units (declared when present; the symbol test in
# tests/test_abi.py checks that everything include/b200gs.h names is exported)
_OPTIONAL = {}


def register(name, restype, argtypes):
    _OPTIONAL[name] = (restype, argtypes)
    if _lib is not None and hasattr(_lib, name):
        fn = getattr(_lib, name)
        fn.restype = restype
        fn.argtypes = argtypes


def check(rc, what=""):
    if rc != 0:
        msg = lib().b200gs_last_error().decode("utf-8", "replace")
        raise B200GSError(f"{what}: {msg}" if what else msg)


def ptr(t):
    """Device (or host) pointer of a tensor; None / empty tensor -> NULL, like the empty
    tensors the reference passes for absent optional inputs."""
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()


def current_stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


class CallTimer:
    """Times every libb200gs entry point that launches kernels with CUDA events on torch's current stream
    (the stream every kernel of the library is launched on). bench.py keeps it active over the timed region
    to get each kernel family's average duration and launch count; nothing else uses it."""
    # kernels launched per call (for the launch count): see csrc/api.cu and the per-file launchers
    KERNELS = {"b200gs_rast_forward_stage1": 7, "b200gs_rast_forward_stage2": 7, "b200gs_rast_backward": 2, "b200gs_rast_backward_accumulate_sh": 2,
               "b200gs_hexplane_order": 6, "b200gs_hexplane_forward": 1, "b200gs_hexplane_forward_masked": 1, "b200gs_hexplane_backward_masked": 1, "b200gs_hexplane_time_forward": 1, "b200gs_hexplane_time_backward": 1, "b200gs_hexplane_backward": 1, "b200gs_hexplane_regulation": 1,
               "b200gs_deform_mlp_forward": 1, "b200gs_deform_mlp_backward": 1, "b200gs_deform_heads_forward": 1, "b200gs_deform_heads_backward": 1,
               "b200gs_adam_multi": 1, "b200gs_adam_sh": 1,
               "b200gs_activations_forward": 1, "b200gs_activations_backward": 1, "b200gs_l1_loss_fwd_bwd": 1, "b200gs_l1_loss_fwd_bwd_u8": 1,
               "b200gs_ssim_fwd_bwd": 3, "b200gs_ssim_fwd_bwd_u8": 3,   # forward, backward, sum (the trainer always asks for the gradient)
               "b200gs_gather_rows_multi": 1, "b200gs_dist2": 8, "b200gs_mark_visible": 1, "b200gs_sort_pairs_u32": 6}

    def __init__(self):
        self.events = {}
        self._orig = {}

    def __enter__(self):
        import torch
        L = lib()
        for name in self.KERNELS:
            if not hasattr(L, name):
                continue
            orig = getattr(L, name)
            self._orig[name] = orig
            rec = self.events.setdefault(name, [])

            def wrapped(*a, _orig=orig, _rec=rec):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = _orig(*a)
                e1.record()
                _rec.append((e0, e1))
                return r
            setattr(L, name, wrapped)
        return self

    def __exit__(self, *exc):
        L = lib()
        for name, orig in self._orig.items():
            setattr(L, name, orig)
        self._orig = {}

    def reset(self):
        for v in self.events.values():
            v.clear()

    def summary(self):
        """{entry: {"calls", "ms_total", "ms_avg", "kernels"}} — call after a device synchronize."""
        out = {}
        for name, ev in self.events.items():
            if not ev:
                continue
            ms = [a.elapsed_time(b) for a, b in ev]
            out[name] = {"calls": len(ms), "ms_total": sum(ms), "ms_avg": sum(ms) / len(ms), "kernels": self.KERNELS[name] * len(ms)}
        return out
