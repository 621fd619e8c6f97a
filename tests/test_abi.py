"""CPU: the C-ABI library loads without a GPU and exports every symbol include/b200gs.h
declares; host-side logic (buffer sizing, argument validation, error strings) behaves."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "b200gs.h")


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(b200gs_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from b200gs import _lib
    L = _lib.lib()
    syms = _declared_symbols()
    assert len(syms) >= 15, syms
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    assert L.b200gs_version() >= 100


def test_buffer_sizes_and_errors_without_gpu():
    from b200gs import _lib
    L = _lib.lib()
    out = (ctypes.c_size_t * 3)()
    assert L.b200gs_rast_buffer_sizes(1000, 5000, 640, 480, out) == 0
    g1, b1, i1 = list(out)
    assert L.b200gs_rast_buffer_sizes(2000, 10000, 1280, 720, out) == 0
    g2, b2, i2 = list(out)
    assert g2 > g1 and b2 > b1 and i2 > i1 and all(v % 256 == 0 for v in (g1, b1, i1))
    assert g1 >= 1000 * 75          # at least the per-Gaussian state the reference keeps (rasterizer_impl.h:21-37)
    assert L.b200gs_rast_buffer_sizes(-1, 0, 640, 480, out) != 0
    assert b"bad arguments" in L.b200gs_last_error()
    assert L.b200gs_rast_buffer_sizes(0, 0, 16, 16, out) == 0      # empty scene is legal
    assert L.b200gs_sort_temp_bytes(1 << 20, 0, 32) > L.b200gs_sort_temp_bytes(1 << 10, 0, 32)
    assert L.b200gs_dist2_scratch_bytes(1000) > 1000 * 32


def test_product_path_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "iclr2025_3d-mom_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("Oracle", ""), os.path.join(dirpath, f)


def test_cpu_tensors_are_rejected_loudly():
    import torch
    from b200gs.rasterizer import _C
    from b200gs.knn import distCUDA2
    with pytest.raises(RuntimeError):
        distCUDA2(torch.zeros(10, 3))
    with pytest.raises(RuntimeError):
        _C.rasterize_gaussians(torch.zeros(3), torch.zeros(5, 2), torch.Tensor([]), torch.zeros(5, 1), torch.zeros(5, 3),
                               torch.zeros(5, 4), 1.0, torch.Tensor([]), torch.eye(4), torch.eye(4), 1.0, 1.0, 16, 16,
                               torch.zeros(5, 16, 3), 3, torch.zeros(3), False, False)


def test_dropin_modules_expose_reference_names():
    import diff_gaussian_rasterization as dgr
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer  # noqa: F401
    assert GaussianRasterizationSettings._fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg",
                                                     "scale_modifier", "viewmatrix", "projmatrix", "sh_degree", "campos",
                                                     "prefiltered", "debug")
    for name in ("rasterize_gaussians", "_RasterizeGaussians", "_C"):
        assert hasattr(dgr, name)
    from diff_gaussian_rasterization import _C as c_mod
    for name in ("rasterize_gaussians", "rasterize_gaussians_backward", "mark_visible"):
        assert hasattr(c_mod, name)
    from simple_knn._C import distCUDA2  # noqa: F401


def test_call_timer_table_names_are_abi_entries():
    """bench.py's per-entry-point timing wraps libb200gs functions by name: every name must be a declared, exported entry."""
    import re
    from b200gs import _lib
    header = open(os.path.join(ROOT, "include", "b200gs.h")).read()
    declared = set(re.findall(r"\b(b200gs_[a-z0-9_]+)\s*\(", header))
    L = _lib.lib()
    for name in _lib.CallTimer.KERNELS:
        assert name in declared, name
        assert hasattr(L, name), name


RETIRED_OPTIONS = (b"mlp_bwd_v2", b"mlp_fwd_elect", b"mlp_bwd_ablate", b"hexplane_time_fwd", b"hexplane_time_bwd",
                   b"lookback_parallel", b"sort_ballot_rank", b"composite_pairs", b"sort_small_tiles", b"sort_balanced_digits")


def test_launch_settings_and_retired_option_names():
    """Launch settings (include/b200gs.h: b200gs_set_option): the two MLP SM caps round-trip from their default 0; the
    kernel-generation switches of earlier rounds are unknown names; the environment changes nothing."""
    import subprocess
    import sys
    from b200gs import _lib
    L = _lib.lib()
    for name in (b"mlp_fwd_sms", b"mlp_bwd_sms"):
        assert L.b200gs_get_option(name) == 0
        assert L.b200gs_set_option(name, 120) == 0 and L.b200gs_get_option(name) == 120
        assert L.b200gs_set_option(name, 0) == 0 and L.b200gs_get_option(name) == 0
    for name in RETIRED_OPTIONS + (b"no_such_option",):
        assert L.b200gs_get_option(name) == -1, name
        assert L.b200gs_set_option(name, 1) != 0 and b"unknown option" in L.b200gs_last_error(), name
        assert L.b200gs_get_option(name) == -1, name
    # the library reads no environment variables: a process started with the old B200GS_* switches sees the same answers
    names = [n.decode() for n in (b"mlp_fwd_sms", b"mlp_bwd_sms") + RETIRED_OPTIONS]
    probe = ("import ctypes, sys; L = ctypes.CDLL(sys.argv[1]); "
             "print([L.b200gs_get_option(n.encode()) for n in sys.argv[2:]])")
    env = dict(os.environ, B200GS_MLP_BWD_V2="0", B200GS_MLP_FWD_ELECT="0", B200GS_MLP_FWD_SMS="100",
               B200GS_MLP_BWD_SMS="100", B200GS_COMPOSITE_PAIRS="0", B200GS_SORT_BALLOT_RANK="0", B200GS_PROFILING="1")
    r = subprocess.run([sys.executable, "-c", probe, _lib.LIB_PATH] + names, env=env, capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == str([0, 0] + [-1] * len(RETIRED_OPTIONS))


def test_mlp_backward_refuses_misaligned_weight_gradients():
    """The tcgen05 MLP backward (feat_dim 64) flushes the W1 / W2 gradients with 128-bit reductions: a gradient pointer
    that is not 16-byte aligned is an error raised before anything touches the device."""
    from b200gs import _lib
    from b200gs.field import _MlpGrads, _MlpWeights
    L = _lib.lib()
    w = _MlpWeights(feat_dim=64, width=64, w1=0x10000, b1=0x20000)
    for h in range(3):
        w.w2[h], w.b2[h], w.w3[h], w.b3[h] = 0x30000 + 0x1000 * h, 0x40000, 0x50000, 0x60000
    for bad in ("w1", "w2"):
        gw = _MlpGrads(w1=0x70000, b1=0x80000)
        for h in range(3):
            gw.w2[h], gw.b2[h], gw.w3[h], gw.b3[h] = 0x90000 + 0x1000 * h, 0xa0000, 0xb0000, 0xc0000
        if bad == "w1":
            gw.w1 = 0x70004
        else:
            gw.w2[1] = 0x91008
        rc = L.b200gs_deform_mlp_backward(ctypes.byref(w), ctypes.byref(gw), ctypes.c_longlong(1000), None, None, None,
                                          None, None, None, None)
        assert rc != 0, bad
        assert b"16-byte aligned" in L.b200gs_last_error(), (bad, L.b200gs_last_error())
