"""Times the HexPlane grid as the reference's own Deformation runs it once b200gs.launcher.patch_hexplane has put
b200gs.field.HexPlaneField in its place, against the reference's PyTorch grid (F.grid_sample + autograd, float32).  Prints one
JSON line.

    python tools/time_hexplane_channels.py [--reps 20] [--out profiles/x.json]

  * configurations: 16 channels at 2 and 3 levels and, as the control, 32 channels at 2 levels; spatial resolution 64 m
    (m = 1, 2, 4 per level), time resolution 150; P = 262,144 (the reference pipeline's size) and 1,048,576.
  * the call as the reference makes it: every call hands the grid a fresh [P, 63] encoding's [:, :3] slice and the view's one
    timestamp as a [P, 1] tensor, so each call copies xyz, checks the timestamp for uniformity (one 8-byte read-back), re-sorts
    the points by cell (b200gs_hexplane_order; P >= 16,384) and runs the six-plane kernel; its backward runs the six-plane
    backward (at 16 channels with the time planes' gradient reduced through replicated 1-D rows).  The tool checks that
    every timed call sorted (b200gs._lib.COUNTERS["cell_order_sorts"]).  `order_ms` is the sort alone; `order_share` =
    order_ms / fused forward.
  * `kernel_*_ms`: the forward / backward kernels alone through the C ABI (cell order precomputed, uniform timestamp).
  * torch: oracle/field_torch.py hexplane_features (the reference's interpolate_ms_features) on contiguous float32 planes;
    forward, and forward + autograd backward (xyz and plane gradients).
  * traffic model (bytes per point, not measured): forward reads xyz 12 + order 4 and writes C levels 4 of features;
    backward reads xyz 12 + order 4 + d_features C levels 4 and writes d_xyz 12; the planes (and their gradients, read and
    written once) are added amortised over P.  Texel gathers beyond the first touch are assumed to hit L1 / L2.  `frac_copy`
    = (bytes / kernel time) over the device-to-device copy rate measured in the same process.
  * composed: a stand-in for the reference's Deformation at dynerf width 128 (tools/hexplane_standins.py StandInDeformation,
    the module tests/test_hexplane_channels.py checks) over our grid and over the PyTorch grid, forward + backward of all five
    heads (one sort per call as well).
CUDA events around every call; the 126 MB L2 is overwritten (256 MB memset, not timed) before each call.
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "iclr2025_3d-mom_b200"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)

import torch

from hexplane_standins import StandInDeformation, TorchGrid
from time_ssim import gpu_info, hbm_peak, timed

CONFIGS = ((16, 2), (16, 3), (32, 2))
SIZES = (262144, 1 << 20)


def _grid(C, levels):
    from b200gs import field
    torch.manual_seed(0)
    cfg = {'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': C, 'resolution': [64, 64, 64, 150]}
    f = field.HexPlaneField(1.6, cfg, [1, 2, 4][:levels]).cuda()
    with torch.no_grad():
        for p in f._planes():
            p.add_(torch.randn_like(p) * 0.1)
    return f


def timed_sorting(fn, reps, flush):
    """timed() over calls that must each sort the points once (3 warm-up calls + reps)."""
    from b200gs import _lib
    before = _lib.COUNTERS["cell_order_sorts"]
    ms = timed(fn, reps, flush)
    sorts = _lib.COUNTERS["cell_order_sorts"] - before
    if sorts != reps + 3:
        raise SystemExit(f"expected one cell sort per call, counted {sorts} over {reps + 3} calls")
    return ms


def one(C, levels, P, reps, flush, copy_gbs):
    from b200gs import _lib, field
    from b200gs._lib import current_stream
    L = _lib.lib()
    f = _grid(C, levels)
    g = torch.Generator(device="cuda").manual_seed(1)
    emb = torch.rand(P, 63, device="cuda", generator=g) * 3.2 - 1.6
    t = torch.full((P, 1), 0.37, device="cuda")
    F = C * levels
    dfeat = torch.randn(P, F, device="cuda", generator=g)
    r = {"channels": C, "levels": levels, "P": P}

    # the call as the reference's Deformation makes it
    def fused_fwd():
        return f(emb[:, :3], t)
    r["fused_fwd_ms"] = timed_sorting(fused_fwd, reps, flush)
    x = emb[:, :3].detach().requires_grad_(True)
    feat = f(x, t)

    def fused_bwd():
        torch.autograd.backward(feat, dfeat, retain_graph=True)
    r["fused_bwd_ms"] = timed(fused_bwd, reps, flush)
    xyz = emb[:, :3].contiguous()
    order = torch.empty(P, dtype=torch.int32, device="cuda")
    nbytes = L.b200gs_hexplane_order_scratch_bytes(P)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    r["order_ms"] = timed(lambda: L.b200gs_hexplane_order(P, xyz.data_ptr(), f.aabb.data_ptr(), order.data_ptr(), scratch.data_ptr(),
                                                          nbytes, current_stream()), reps, flush)
    r["order_share"] = r["order_ms"] / r["fused_fwd_ms"]

    # the kernels alone
    planes, res = f._planes(), tuple(f._res)
    grads = [torch.zeros_like(p, memory_format=torch.preserve_format) for p in planes]
    d = field._hex_desc(f.aabb, planes, levels, res, grads)
    out = torch.empty(P, F, device="cuda")
    d_xyz = torch.empty(P, 3, device="cuda")
    rows, rbytes = field._time_row_scratch(d, xyz.device)
    use_rows = C == 16                       # what HexPlaneField's backward does with one timestamp
    r["kernel_fwd_ms"] = timed(lambda: L.b200gs_hexplane_forward_masked(ctypes.byref(d), P, xyz.data_ptr(), order.data_ptr(), None, 0.37,
                                                                        0x3F, None, out.data_ptr(), current_stream()), reps, flush)
    r["kernel_bwd_ms"] = timed(lambda: L.b200gs_hexplane_backward_masked(
        ctypes.byref(d), P, xyz.data_ptr(), order.data_ptr(), None, 0.37, 0x3F, None, None, dfeat.data_ptr(), d_xyz.data_ptr(),
        rows.data_ptr() if use_rows else None, rbytes if use_rows else 0, current_stream()), reps, flush)
    plane_bytes = sum(p.numel() for p in planes) * 4
    fwd_b = 12 + 4 + 4 * F + plane_bytes / P
    bwd_b = 12 + 4 + 4 * F + 12 + 3 * plane_bytes / P
    r["bytes_per_point"] = {"fwd": round(fwd_b, 1), "bwd": round(bwd_b, 1)}
    r["frac_copy"] = {"fwd": fwd_b * P / (r["kernel_fwd_ms"] * 1e-3) / 1e9 / copy_gbs,
                      "bwd": bwd_b * P / (r["kernel_bwd_ms"] * 1e-3) / 1e9 / copy_gbs}

    # the reference's PyTorch grid, float32
    tg = TorchGrid(f, torch.float32)
    with torch.no_grad():
        r["torch_fwd_ms"] = timed(lambda: tg(emb[:, :3], t), reps, flush)

    def torch_fwd_bwd():
        xx = emb[:, :3].detach().requires_grad_(True)
        torch.autograd.backward(tg(xx, t), dfeat)
    r["torch_fwd_bwd_ms"] = timed(torch_fwd_bwd, reps, flush)

    def fused_fwd_bwd():
        xx = emb[:, :3].detach().requires_grad_(True)
        torch.autograd.backward(f(xx, t), dfeat)
    r["fused_fwd_bwd_ms"] = timed_sorting(fused_fwd_bwd, reps, flush)
    r["torch_over_fused_fwd_bwd"] = r["torch_fwd_bwd_ms"] / r["fused_fwd_bwd_ms"]
    return r


def composed(C, levels, P, reps, flush):
    f = _grid(C, levels)
    torch.manual_seed(2)
    ours = StandInDeformation(f).cuda()
    ref = StandInDeformation(TorchGrid(f, torch.float32)).cuda().copy_mlp_from(ours)
    g = torch.Generator(device="cuda").manual_seed(3)
    emb = torch.rand(P, 63, device="cuda", generator=g) * 3.2 - 1.6
    t = torch.full((P, 1), 0.37, device="cuda")
    ws = [torch.randn(P, k, device="cuda", generator=g) for _, k in StandInDeformation.HEADS]

    def step(m):
        e = emb.detach().requires_grad_(True)
        torch.autograd.backward(m(e, t), ws)
    r = {"channels": C, "levels": levels, "P": P, "width": 128,
         "ours_fwd_bwd_ms": timed_sorting(lambda: step(ours), reps, flush), "torch_fwd_bwd_ms": timed(lambda: step(ref), reps, flush)}
    r["torch_over_ours"] = r["torch_fwd_bwd_ms"] / r["ours_fwd_bwd_ms"]
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_hexplane_channels.py measures on a CUDA device; none is visible")
    gpu = gpu_info()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    copy_gbs = hbm_peak()
    res = {"gpu": gpu, "copy_GBps": copy_gbs, "reps": a.reps, "grid": [one(C, lv, P, a.reps, flush, copy_gbs) for P in SIZES for C, lv in CONFIGS],
           "composed": [composed(C, lv, P, a.reps, flush) for P in SIZES for C, lv in ((16, 2), (32, 2))]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
