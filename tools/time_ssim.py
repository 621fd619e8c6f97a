"""Times the fused SSIM value + gradient (csrc/ssim.cu) against the reference's PyTorch formulation, and one trainer step with
and without the D-SSIM term.  Prints one JSON line.

    python tools/time_ssim.py [--reps 50]

  * fused: one [3,H,W] view, forward + backward (the two launches of fusedops.dssim_loss_and_grad), and the value-only forward,
    at 1280x720, 1920x1080 and 3840x2160.  CUDA events around each call; the 126 MB L2 is overwritten (256 MB memset, not
    timed) before every call, so inputs come from HBM as they do after the rasterizer in a training step.
  * torch: utils/loss_utils.py:ssim restated in PyTorch (oracle/ssim_torch.py), float32, forward + autograd backward with
    respect to the render, with cuDNN's default TF32 setting and with TF32 off, same L2 treatment.
  * hbm_peak_gbs: a device-to-device copy of 1 GiB measured in the same process (read + write bytes over time).
  * traffic model: the two-launch design moves 48 B per pixel and channel (forward reads x, y and writes A, B, Cc; backward
    reads A, B, Cc, x, y, d and writes d); a single fused pass would need 16 B (x, y, d read, d written).
  * trainer: ViewParallelTrainer.step over 2 views of 1280x720 with 200k Gaussians, lambda_dssim 0 and 0.2 (ms per step).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "iclr2025_3d-mom_b200"), os.path.join(ROOT, "iclr2025_3d-mom_b200", "dropin")):
    sys.path.insert(0, p)

import torch


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed(fn, reps, flush):
    """Mean milliseconds of fn() over reps calls, each after overwriting L2 (the overwrite is outside the events)."""
    for _ in range(3):
        fn()
    ms = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        ms.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ms) / reps


def hbm_peak(gib=1):
    src = torch.empty(gib << 28, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        dst.copy_(src)
    b.record()
    torch.cuda.synchronize()
    return 2 * src.numel() * 4 * 20 / (a.elapsed_time(b) * 1e-3) / 1e9


def trainer_step_ms(lambda_dssim, steps=10, P=200000, W=1280, H=720):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    raw = syn.make_gaussians(P, scale_mu=0.01, seed=3, device="cpu")
    torch.manual_seed(0)
    m = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}).to(dev)
    m.training_setup()
    tr = engine.ViewParallelTrainer(m, torch.zeros(3, device=dev), stage="fine", lambda_dssim=lambda_dssim)
    cams = syn.orbit_cameras(2, W, H, device=dev)
    g = torch.Generator().manual_seed(1)
    gts = [torch.rand(3, H, W, generator=g).to(dev) for _ in cams]
    for _ in range(3):
        tr.step(cams, gts)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        loss = tr.step(cams, gts)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps, float(loss)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_ssim.py measures on the GPU; there is no CPU path")
    from b200gs import fusedops
    from oracle import ssim_torch
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > L2
    res = {"tool": "time_ssim", "gpu": gpu_info(), "reps": args.reps, "l2": "overwritten before every timed call"}
    res["hbm_peak_gbs"] = round(hbm_peak(), 1)
    sizes = {}
    for W, H in ((1280, 720), (1920, 1080), (3840, 2160)):
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.rand(3, H, W, device="cuda", generator=g)
        y = torch.rand(3, H, W, device="cuda", generator=g)
        loss = torch.zeros(1, device="cuda")
        d = torch.zeros_like(x)
        sums = torch.zeros(1, device="cuda")
        row = {}
        row["fused_fwd_bwd_us"] = 1e3 * timed(lambda: fusedops.dssim_loss_and_grad(x, y, 0.2, loss, d), args.reps, flush)
        row["fused_value_only_us"] = 1e3 * timed(lambda: fusedops._ssim_launch(x[None], y[None], 0.0, 1.0, sums, 0.0, None),
                                                 args.reps, flush)

        def torch_ref():
            xr = x[None].detach().requires_grad_(True)
            (0.2 * (1.0 - ssim_torch.ssim(xr, y[None]))).backward()
        prev = torch.backends.cudnn.allow_tf32
        try:
            torch.backends.cudnn.allow_tf32 = True
            row["torch_tf32_default_us"] = 1e3 * timed(torch_ref, max(10, args.reps // 5), flush)
            torch.backends.cudnn.allow_tf32 = False
            row["torch_tf32_off_us"] = 1e3 * timed(torch_ref, max(10, args.reps // 5), flush)
        finally:
            torch.backends.cudnn.allow_tf32 = prev
        n = 3 * H * W
        row["traffic_mb"] = round(48 * n / 1e6, 2)
        row["achieved_gbs"] = round(48 * n / (row["fused_fwd_bwd_us"] * 1e-6) / 1e9, 1)
        row["fraction_of_measured_hbm_peak"] = round(row["achieved_gbs"] / res["hbm_peak_gbs"], 3)
        row["single_pass_bound_us"] = round(16 * n / (res["hbm_peak_gbs"] * 1e9) * 1e6, 2)
        row["speedup_vs_torch_tf32_default"] = round(row["torch_tf32_default_us"] / row["fused_fwd_bwd_us"], 1)
        row["speedup_vs_torch_tf32_off"] = round(row["torch_tf32_off_us"] / row["fused_fwd_bwd_us"], 1)
        for k in ("fused_fwd_bwd_us", "fused_value_only_us", "torch_tf32_default_us", "torch_tf32_off_us"):
            row[k] = round(row[k], 2)
        sizes[f"{W}x{H}"] = row
        del x, y, d
    res["per_view"] = sizes
    t0, l0 = trainer_step_ms(0.0)
    t2, l2 = trainer_step_ms(0.2)
    res["trainer_step_ms"] = {"views": 2, "size": "1280x720", "gaussians": 200000, "lambda_dssim_0": round(t0, 3),
                              "lambda_dssim_0.2": round(t2, 3), "loss_0": l0, "loss_0.2": l2}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
