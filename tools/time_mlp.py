"""Deformation-MLP kernels alone (C3 point count): device time per launch of b200gs_deform_mlp_forward / _backward through the
C ABI, CUDA events on the launching stream, L2 flushed by the working set itself (1.4 / 1.6 GB per launch).  Knobs:
    P = point count (default 1000000)
    MULTIRES = HexPlane level multipliers (default 1,2: 2 levels, feature dim 64, the reference's configuration;
               1,2,4,8: 4 levels, feature dim 128)
    python tools/time_mlp.py
    MULTIRES=1,2,4,8 P=1000000 python tools/time_mlp.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in ("iclr2025_3d-mom_b200", "tests", ""):
    sys.path.insert(0, os.path.join(ROOT, p))
import torch

import test_field_parity as T

P = int(os.environ.get("P", 1000000))
MULTIRES = [int(m) for m in os.environ.get("MULTIRES", "1,2").split(",")]
net = T._model(MULTIRES, 50)
xyz, scales, rot, opacity, shs, flow = T._inputs(P)
frame_num = torch.tensor(22, device="cuda")
a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
g = torch.Generator().manual_seed(5)
w = [torch.randn(P, k, generator=g).cuda() for k in (3, 3, 4)]
from torch.profiler import ProfilerActivity, profile


def step():
    pts, sc, rt, _, _ = net(a[0], a[1], a[2], opacity, shs, 0.37, flow, frame_num, 1)
    ((pts * w[0]).sum() + (sc * w[1]).sum() + (rt * w[2]).sum()).backward()


for _ in range(3):
    step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(10):
        step()
    torch.cuda.synchronize()
rows = [(e.key, e.device_time_total / max(e.count, 1), e.count) for e in prof.key_averages() if "deform_mlp" in e.key or "hexplane" in e.key]
print(f"P = {P}, multires = {MULTIRES}")
for k, us, n in sorted(rows, key=lambda r: -r[1]):
    print(f"{us:9.1f} us x{n:3d}  {k[:100]}")
