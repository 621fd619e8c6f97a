"""Times the opacity / SH deformation-head kernels (csrc/deform_heads.cu) against the same two heads as PyTorch ops, and one
trainer step with the heads off and on.  Prints one JSON line.

    python tools/time_deform_heads.py [--reps 50] [--P 1000000]

  * kernels: b200gs_deform_heads_forward / _backward through the C ABI at P points, feature dim 64, tiled features (the
    layout the trainer's one-timestamp views use), both heads on, the backward adding d shs into an SH gradient buffer
    (written, as on a step's first view).  CUDA events around each call; the 126 MB L2 is overwritten (256 MB memset, not
    timed) before every call.
  * torch: ReLU, Linear(64,64), ReLU, Linear(64,k) for k = 1 and 48 on the same relu(hidden) plus the two adds, float32 with
    TF32 off (torch's default for matmuls), forward alone and forward + autograd backward (hidden, weights, biases).
  * traffic model (bytes per point, not measured): forward reads relu(hidden) 256, opacity 4, shs 192 and writes
    relu(z) 2 x 256, opacity' 4, shs' 192 = 1160; backward reads relu(hidden) 256, relu(z) 512, d opacity' 4, d shs' 192,
    features 256, reads and writes d_features 2 x 256 and writes d shs 192 = 1924.  Achieved fraction = (bytes / time) over
    the device-to-device copy rate measured in the same process.
  * trainer: ViewParallelTrainer.step over 2 views of 1280x720 with 200k Gaussians, no_do = no_dshs = True and both False.
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "iclr2025_3d-mom_b200"), os.path.join(ROOT, "iclr2025_3d-mom_b200", "dropin"),
          os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)

import torch

from time_ssim import gpu_info, hbm_peak, timed

FWD_BYTES, BWD_BYTES = 1160, 1924


def kernel_times(P, reps, flush):
    from b200gs import _lib
    from b200gs.field import _HeadsGrads, _HeadsWeights, _MlpWeights
    L = _lib.lib()
    dev = torch.device("cuda")
    stream = lambda: torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(0)
    F, MW = 64, 64
    lin = lambda o, i: ((torch.rand(o, i, generator=g, device=dev) * 2 - 1) / i ** 0.5, torch.randn(o, generator=g, device=dev) * 0.05)
    w1, b1 = lin(MW, F)
    geo = [lin(MW, MW) + lin(k, MW) for k in (3, 3, 4)]
    heads = [lin(MW, MW) + lin(k, MW) for k in (1, 48)]
    n_tiles = (P + 127) // 128
    feat = torch.randn(n_tiles * 128 * MW, generator=g, device=dev) * 0.6 + 0.15          # tiled layout
    saved = torch.empty(L.b200gs_deform_mlp_saved_floats(P), device=dev)
    ins = [torch.zeros(P, k, device=dev) for k in (3, 3, 4, 3)]
    outs = [torch.empty(P, k, device=dev) for k in (3, 3, 4)]
    mw = _MlpWeights(feat_dim=F, width=MW, w1=w1.data_ptr(), b1=b1.data_ptr(), feat_tiled=1)
    for h in range(3):
        mw.w2[h], mw.b2[h], mw.w3[h], mw.b3[h] = (t.data_ptr() for t in geo[h])
    assert L.b200gs_deform_mlp_forward(ctypes.byref(mw), P, feat.data_ptr(), *[t.data_ptr() for t in ins], 0.0, None, 0.0,
                                       *[t.data_ptr() for t in outs], saved.data_ptr(), stream()) == 0
    hw = _HeadsWeights(feat_dim=F, width=MW, w1=w1.data_ptr(), feat_tiled=1)
    for h in range(2):
        hw.w2[h], hw.b2[h], hw.w3[h], hw.b3[h] = (t.data_ptr() for t in heads[h])
    op, shs = torch.randn(P, 1, generator=g, device=dev), torch.randn(P, 16, 3, generator=g, device=dev)
    op_o, shs_o = torch.empty_like(op), torch.empty_like(shs)
    hs = torch.empty(L.b200gs_deform_heads_saved_floats(P), device=dev)
    d_op, d_sh = torch.randn_like(op), torch.randn_like(shs)
    d_feat = torch.zeros_like(feat)
    sh_grad = torch.empty_like(shs)
    gbufs = [torch.zeros(MW, F, device=dev), torch.zeros(MW, device=dev)] + [torch.zeros_like(t) for hd in heads for t in hd]
    hg = _HeadsGrads(w1=gbufs[0].data_ptr(), b1=gbufs[1].data_ptr())
    for h in range(2):
        hg.w2[h], hg.b2[h], hg.w3[h], hg.b3[h] = (t.data_ptr() for t in gbufs[2 + 4 * h: 6 + 4 * h])

    def fwd():
        assert L.b200gs_deform_heads_forward(ctypes.byref(hw), P, 16, saved.data_ptr(), op.data_ptr(), shs.data_ptr(),
                                             op_o.data_ptr(), shs_o.data_ptr(), hs.data_ptr(), stream()) == 0

    def bwd():
        assert L.b200gs_deform_heads_backward(ctypes.byref(hw), ctypes.byref(hg), P, 16, feat.data_ptr(), saved.data_ptr(),
                                              hs.data_ptr(), d_op.data_ptr(), d_sh.data_ptr(), d_feat.data_ptr(),
                                              sh_grad.data_ptr(), 1, stream()) == 0
    t_fwd, t_bwd = timed(fwd, reps, flush), timed(bwd, reps, flush)

    # the same heads as PyTorch ops
    idx = (torch.arange(P, device=dev)[:, None] >> 7) * (128 * MW) + ((torch.arange(P, device=dev)[:, None] & 127) >> 2) * 256 \
        + (torch.arange(MW, device=dev)[None, :] >> 2) * 16 + (torch.arange(P, device=dev)[:, None] & 3) * 4 + (torch.arange(MW, device=dev)[None, :] & 3)
    hidden = saved[idx].contiguous()
    params = [t.clone().requires_grad_(True) for hd in heads for t in hd]

    def torch_fwd(grad):
        hd = hidden.clone().requires_grad_(grad)
        outs = []
        for h, base in enumerate((op, shs.reshape(P, 48))):
            w2, b2, w3, b3 = params[4 * h: 4 * h + 4]
            z = torch.relu(torch.nn.functional.linear(torch.relu(hd), w2, b2))
            outs.append(base * 1 + torch.nn.functional.linear(z, w3, b3))
        if grad:
            torch.autograd.backward(outs, [d_op, d_sh.reshape(P, 48)])
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            t_tf = timed(lambda: torch_fwd(False), max(10, reps // 5), flush)
        t_tfb = timed(lambda: torch_fwd(True), max(10, reps // 5), flush)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return t_fwd, t_bwd, t_tf, t_tfb


def trainer_step_ms(no_heads, steps=10, P=200000, W=1280, H=720):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    raw = syn.make_gaussians(P, scale_mu=0.01, seed=3, device="cpu")
    torch.manual_seed(0)
    h = engine.default_hyper()
    h.no_do = h.no_dshs = no_heads
    m = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}, hyper=h).to(dev)
    m.training_setup()
    tr = engine.ViewParallelTrainer(m, torch.zeros(3, device=dev), stage="fine")
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
    ap.add_argument("--P", type=int, default=1000000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_deform_heads.py measures on the GPU; there is no CPU path")
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")          # 256 MB > L2
    res = {"tool": "time_deform_heads", "gpu": gpu_info(), "reps": args.reps, "P": args.P, "feat_dim": 64, "feat_tiled": 1,
           "l2": "overwritten before every timed call"}
    peak = hbm_peak()
    res["hbm_copy_peak_gbs"] = round(peak, 1)
    t_fwd, t_bwd, t_tf, t_tfb = kernel_times(args.P, args.reps, flush)
    for name, t, nbytes in (("forward", t_fwd, FWD_BYTES), ("backward", t_bwd, BWD_BYTES)):
        gbs = nbytes * args.P / (t * 1e-3) / 1e9
        res[name] = {"us": round(1e3 * t, 1), "bytes_per_point_model": nbytes, "achieved_gbs": round(gbs, 1),
                     "fraction_of_copy_peak": round(gbs / peak, 3),
                     "bound_us_at_copy_peak": round(nbytes * args.P / (peak * 1e9) * 1e6, 1)}
    res["torch_fp32"] = {"forward_us": round(1e3 * t_tf, 1), "forward_backward_us": round(1e3 * t_tfb, 1)}
    t_off, l_off = trainer_step_ms(True)
    t_on, l_on = trainer_step_ms(False)
    res["trainer_step_ms"] = {"views": 2, "size": "1280x720", "gaussians": 200000, "heads_off": round(t_off, 3),
                              "heads_on": round(t_on, 3), "loss_off": l_off, "loss_on": l_on}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
