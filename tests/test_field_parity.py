"""GPU parity: fused HexPlane + deformation-MLP kernels (through the drop-in nn.Modules) against
the plain-PyTorch restatement of the reference modules (oracle/field_torch.py; F.grid_sample +
F.linear on the same device). Tolerances: forward 2e-5 relative to the tensor's max-abs (FP32
accumulation order differs from cuBLAS), gradients 1e-3 relative (north_star)."""
import types

import pytest
import torch

from oracle import field_torch as oracle

pytestmark = pytest.mark.gpu


def _args(multires, T, no_dx=False, no_ds=False, no_dr=False):
    return types.SimpleNamespace(
        net_width=64, timebase_pe=4, defor_depth=0, posebase_pe=10, scale_rotation_pe=2, opacity_pe=2,
        timenet_width=64, timenet_output=32, bounds=1.6, grid_pe=0,
        kplanes_config={'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': 32,
                        'resolution': [64, 64, 64, T]},
        multires=multires, no_dx=no_dx, no_grid=False, no_ds=no_ds, no_dr=no_dr, no_do=True, no_dshs=True,
        empty_voxel=False, static_mlp=False, apply_rotation=False)


def _model(multires, T, seed=0, **heads_off):
    from b200gs.field import deform_network
    torch.manual_seed(seed)
    net = deform_network(_args(multires, T, **heads_off)).cuda()
    with torch.no_grad():
        for p in net.deformation_net.grid.grids.parameters():
            p.add_(torch.randn_like(p) * 0.01)       # make the time planes non-trivial (SURVEY §8d)
        for n, p in net.named_parameters():
            if n.endswith("bias"):
                p.add_(torch.randn_like(p) * 0.05)
    net.deformation_net.set_aabb([1.4, 1.3, 1.45], [-1.35, -1.4, -1.2])
    return net


def _inputs(P, seed=1):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(P, 3, generator=g) * 3.4 - 1.7).cuda()           # ~15% outside the aabb -> border clamp
    scales = (torch.randn(P, 3, generator=g) * 0.6 - 5).cuda()
    rot = torch.randn(P, 4, generator=g).cuda()
    opacity = torch.randn(P, 1, generator=g).cuda()
    shs = torch.randn(P, 16, 3, generator=g).cuda()
    flow = (torch.randn(P, 3, generator=g) * 1e-3).cuda()
    return xyz, scales, rot, opacity, shs, flow


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


_FULL = [([1, 2], 50, 1000000)]      # BASELINE.json C3 point count (always on: seconds on a B200)


_CASES = [([1, 2], 50, 5000), ([1, 2], 50, 64), ([1, 2], 50, 1), ([1, 2, 4, 8], 25, 3001),
          ([1, 2], 50, 40003), ([1, 2], 50, -5000), ([1, 2], 50, -40003)] + _FULL      # >= 16384 points: cell-ordered traversal
# disabled heads (no_dx / no_ds / no_dr): pass-through outputs, no stash-free inference, no gradient for the head's parameters
_HEADS_OFF = [{"no_ds": True}, {"no_dx": True, "no_dr": True}]


@pytest.mark.parametrize("multires,T,P,heads_off",
                         [pytest.param(m, T, P, {}, id=f"multires{i}-{T}-{P}") for i, (m, T, P) in enumerate(_CASES)] +
                         [pytest.param(m, T, P, off, id=f"multires{i}-{T}-{P}-" + "-".join(off)) for off in _HEADS_OFF
                          for i, (m, T, P) in enumerate(_CASES) if P in (5000, 3001)])
def test_deform_network_forward_backward(multires, T, P, heads_off):
    # P < 0: |P| points with a DIFFERENT timestamp per point (the general [P,1] tensor of gaussian_renderer/__init__.py:56);
    # otherwise the camera's one timestamp repeated, which field.DETECT_UNIFORM_TIME routes to the one-timestamp kernels
    per_point_time = P < 0
    P = abs(P)
    net = _model(multires, T, **heads_off)
    levels = len(multires)
    xyz, scales, rot, opacity, shs, flow = _inputs(P)
    time = torch.rand(P, 1, generator=torch.Generator().manual_seed(9)).cuda() if per_point_time else torch.full((P, 1), 0.37, device="cuda")
    frame_num = torch.tensor(22, device="cuda")
    sd = {k: v.detach().clone().contiguous().requires_grad_(v.dtype.is_floating_point) for k, v in net.state_dict().items()}

    a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
    pts, sc, rt, op, sh = net(a[0], a[1], a[2], opacity, shs, time, flow, frame_num, 1)
    b = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
    rp, rs, rr, ro, rsh = oracle.deform_forward(sd, levels, b[0], b[1], b[2], opacity, shs, time, flow, frame_num, 1, **heads_off)
    assert _rel(pts, rp) < 2e-5 and _rel(sc, rs) < 2e-5 and _rel(rt, rr) < 2e-5
    assert torch.equal(op, ro) and sh is shs

    g = torch.Generator().manual_seed(5)
    wp, ws, wr = (torch.randn(P, 3, generator=g).cuda(), torch.randn(P, 3, generator=g).cuda(),
                  torch.randn(P, 4, generator=g).cuda())
    ((pts * wp).sum() + (sc * ws).sum() + (rt * wr).sum()).backward()
    ((rp * wp).sum() + (rs * ws).sum() + (rr * wr).sum()).backward()
    for x, y, name in zip(a, b, ("xyz", "scales", "rot")):
        if P < 100000:
            assert _rel(x.grad, y.grad) < 1e-3, name
        else:
            # At a million points a few dozen of the 256M hidden pre-activations sit within FP32 summation-order noise of 0,
            # where two FP32 implementations' ReLU masks legitimately differ and that POINT's gradient changes by a few per
            # cent (tools/debug_hexplane_fullsize.py: the HexPlane kernels alone agree with torch to 4e-7 at this size).
            # Everything else must meet the bar, and the exceptions must stay that rare.
            err = (x.grad - y.grad).abs().max(dim=1).values / y.grad.abs().max()
            bad = err > 1e-3
            assert bad.float().mean().item() < 2e-4, (name, int(bad.sum()))
            assert err[~bad].max().item() < 1e-3
    params = dict(net.named_parameters())
    checked = 0
    worst = 0.0
    if P >= 100000:          # FP64 evaluation of the same oracle: the ground truth both FP32 implementations approximate
        dt = torch.float64
        sd64 = {k: (v.detach().clone().to(dt) if v.dtype.is_floating_point else v.detach().clone()).contiguous().requires_grad_(v.dtype.is_floating_point)
                for k, v in net.state_dict().items()}
        c = [t.clone().to(dt).requires_grad_(True) for t in (xyz, scales, rot)]
        qp, qs, qr, _, _ = oracle.deform_forward(sd64, levels, c[0], c[1], c[2], opacity.to(dt), shs.to(dt), time.to(dt), flow.to(dt), frame_num, 1,
                                                 **heads_off)
        ((qp * wp.to(dt)).sum() + (qs * ws.to(dt)).sum() + (qr * wr.to(dt)).sum()).backward()
    for k, v in sd.items():
        if not v.requires_grad or k.endswith("grid.aabb") or k not in params:
            continue
        p = params[k]
        if v.grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        assert p.grad is not None, k
        if P < 100000:
            worst = max(worst, _rel(p.grad, v.grad))
            assert _rel(p.grad, v.grad) < 1e-3, (k, _rel(p.grad, v.grad))
        else:
            # At this size FP32 itself is not reproducible to 1e-3 of a tensor's scale: torch's own FP32 gradients differ from
            # the same oracle evaluated in FP64 by up to 2e-3 (ReLU-mask flips + summation order; tools/debug_dw_fullsize.py).
            # The meaningful bar is the exact (FP64) gradient: we must be as close to it as the reference's FP32 arithmetic is.
            ref64 = sd64[k].grad
            scale = ref64.abs().max()
            e_ours = ((p.grad.double() - ref64).abs().max() / scale).item()
            e_t32 = ((v.grad.double() - ref64).abs().max() / scale).item()
            assert e_ours <= max(1e-3, 2.0 * e_t32), (k, e_ours, e_t32)
            worst = max(worst, e_ours)
        checked += 1
    print(f"worst parameter-gradient relative error: {worst:.2e}")
    assert checked >= 2 + 4 * (3 - len(heads_off)) + 6 * levels
    # never-used sub-networks get no gradient, exactly like the reference (Appendix C iii)
    assert all(p.grad is None for n, p in net.named_parameters() if n.startswith("timenet") or "opacity_deform" in n or "shs_deform" in n)


def test_hexplane_field_standalone_and_state_dict():
    from b200gs.field import HexPlaneField, deform_network
    torch.manual_seed(3)
    cfg = {'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': 32, 'resolution': [64, 64, 64, 50]}
    f = HexPlaneField(1.6, cfg, [1, 2]).cuda()
    assert f.feat_dim == 64 and f.grids[1][0].shape == (1, 32, 128, 128) and f.grids[0][2].shape == (1, 32, 50, 64)
    P = 777
    g = torch.Generator().manual_seed(4)
    pts = (torch.rand(P, 3, generator=g) * 4 - 2).cuda().requires_grad_(True)
    t = torch.rand(P, 1, generator=g).cuda()
    feat = f(pts, t)
    planes = [p.detach().clone().contiguous().requires_grad_(True) for gp in f.grids for p in gp]
    pts2 = pts.detach().clone().requires_grad_(True)
    ref = oracle.hexplane_features(pts2, t, f.aabb.detach(), planes, 2)
    assert _rel(feat, ref) < 1e-6
    w = torch.randn(P, 64, generator=g).cuda()
    (feat * w).sum().backward(); (ref * w).sum().backward()
    assert _rel(pts.grad, pts2.grad) < 1e-3
    for p, q in zip([p for gp in f.grids for p in gp], planes):
        assert _rel(p.grad, q.grad) < 1e-3
    # state_dict keys / shapes as the reference's checkpoints expect them (SURVEY §5)
    net = deform_network(_args([1, 2], 50))
    keys = set(net.state_dict().keys())
    for k in ["deformation_net.grid.aabb", "deformation_net.grid.grids.0.0", "deformation_net.grid.grids.1.5",
              "deformation_net.feature_out.0.weight", "deformation_net.pos_deform.1.weight",
              "deformation_net.rotations_deform.3.bias", "deformation_net.shs_deform.3.weight", "timenet.0.weight",
              "timenet.2.bias", "time_poc", "pos_poc", "rotation_scaling_poc", "opacity_poc"]:
        assert k in keys, k
    assert len(net.get_grid_parameters()) == 13 and all("grid" not in n for n, _ in net.named_parameters() if False)


def test_inference_forward_without_stash_is_bit_identical():
    """Under torch.no_grad() the MLP forward is told that no backward follows (saved = NULL): nothing is stashed, the outputs
    are the same bits; a backward through such a forward is refused."""
    net = _model([1, 2], 50)
    P = 20011
    xyz, scales, rot, opacity, shs, flow = _inputs(P)
    time = torch.full((P, 1), 0.61, device="cuda")
    fn = torch.tensor(7, device="cuda")
    from b200gs import field
    a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
    keep = field.AUTOGRAD_SPATIAL_SHARING
    field.AUTOGRAD_SPATIAL_SHARING = False          # same HexPlane kernels on both sides: only the stash differs
    try:
        pts, sc, rt, _, _ = net(a[0], a[1], a[2], opacity, shs, time, flow, fn, 1)
    finally:
        field.AUTOGRAD_SPATIAL_SHARING = keep
    with torch.no_grad():
        p2, s2, r2, _, _ = net(xyz, scales, rot, opacity, shs, time, flow, fn, 1)
    assert torch.equal(pts.detach(), p2) and torch.equal(sc.detach(), s2) and torch.equal(rt.detach(), r2)
    assert not p2.requires_grad
    # with the spatial product shared under autograd (the default) the field re-associates the six-plane product: FP32 rounding only
    p3, s3, r3, _, _ = net(a[0], a[1], a[2], opacity, shs, time, flow, fn, 1)
    assert _rel(p3.detach(), p2) < 2e-6 and _rel(s3.detach(), s2) < 2e-6 and _rel(r3.detach(), r2) < 2e-6


def test_autograd_sharing_two_calls_one_backward():
    """field.AUTOGRAD_SPATIAL_SHARING as the reference's training loop meets it: two field calls on the same xyz leaf, then ONE
    backward.  The spatial product is evaluated once, each call samples only its time planes, autograd sums the two calls'
    dL/dS into one spatial backward, and that backward drops the product.  Outputs and gradients equal the same two calls
    without sharing (six-plane forward, MASK_ALL backward per call) up to FP32 re-association."""
    from b200gs import _lib, field
    P = 20011
    xyz, scales, rot, opacity, shs, flow = _inputs(P)
    fn = torch.tensor(7, device="cuda")
    g = torch.Generator().manual_seed(6)
    w = [torch.randn(P, k, generator=g).cuda() for k in (3, 3, 4, 3, 3, 4)]

    def run(share):
        net = _model([1, 2], 50)
        a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
        keep = field.AUTOGRAD_SPATIAL_SHARING
        field.AUTOGRAD_SPATIAL_SHARING = share
        try:
            c0 = _lib.COUNTERS.copy()
            outs = [o for t in (0.2, 0.7) for o in net(a[0], a[1], a[2], opacity, shs, t, flow, fn, 1)[:3]]
            sum((o * wi).sum() for o, wi in zip(outs, w)).backward()
            c1 = _lib.COUNTERS.copy()
            net(a[0], a[1], a[2], opacity, shs, 0.2, flow, fn, 1)
            c2 = _lib.COUNTERS.copy()
        finally:
            field.AUTOGRAD_SPATIAL_SHARING = keep
            field.drop_shared()
        if share:
            assert c1["spatial_product_evaluations"] - c0["spatial_product_evaluations"] == 1
            assert c1["time_row_forward_calls"] - c0["time_row_forward_calls"] == 2
            assert c2["spatial_product_evaluations"] - c1["spatial_product_evaluations"] == 1       # the backward dropped it
        else:
            assert c2["spatial_product_evaluations"] == c0["spatial_product_evaluations"]
        grads = dict(zip(("xyz", "scales", "rot"), (t.grad for t in a)))
        grads.update((n, p.grad) for n, p in net.named_parameters() if p.grad is not None)
        return [o.detach() for o in outs], grads

    shared_outs, shared_grads = run(True)
    plain_outs, plain_grads = run(False)
    for s, p in zip(shared_outs, plain_outs):
        assert _rel(s, p) < 2e-6
    assert shared_grads.keys() == plain_grads.keys() and len(plain_grads) >= 3 + 2 + 12 + 12
    for k, p in plain_grads.items():
        assert _rel(shared_grads[k], p) < 1e-4, k
