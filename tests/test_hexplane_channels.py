"""16-channel HexPlane grids (arguments/dynerf/default.py, arguments/hypernerf/default.py: output_coordinate_dim 16) at 1-4
levels: b200gs.field.HexPlaneField, the six-plane kernels' 16-channel layout (include/b200gs.h b200gs_hexplane_desc.channels),
the launcher's patch_hexplane, and the grid under a stand-in for the reference's own PyTorch Deformation MLP.

GPU bars (as tests/test_hexplane_split_parity.py, anchored on oracle/field_torch.py evaluated in float64): features within
2e-6 and gradients within 1e-4 of each tensor's largest magnitude; the regulariser within 1e-5 (tests/test_regulation_parity.py);
the composed field's MLP part e_ours <= max(1e-3, 2 e_torch32) (DESIGN.md section 5)."""
import ctypes
import itertools
import types

import pytest
import torch

from b200gs import _lib, field
from b200gs.field import _HexDesc
from tools.hexplane_standins import StandInDeformation, TorchGrid

COMBOS = list(itertools.combinations(range(4), 2))


def _cfg(C, res=(64, 48, 40, 150)):
    return {'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': C, 'resolution': list(res)}


def _multires(levels):
    return [1, 2, 4, 8][:levels]


def _hyper(**over):
    from b200gs import engine
    h = engine.default_hyper()
    for k, v in over.items():
        if k == "channels":
            h.kplanes_config = dict(h.kplanes_config, output_coordinate_dim=v)
        else:
            setattr(h, k, v)
    return h


# ---------------------------------------------------------------------------------------------------------------------------
# CPU
@pytest.mark.parametrize("C", [16, 32])
@pytest.mark.parametrize("levels", [1, 2, 3, 4])
def test_field_layout(C, levels):
    res = (6, 5, 7, 9)
    f = field.HexPlaneField(1.6, _cfg(C, res), _multires(levels))
    assert f.feat_dim == C * levels
    sd = f.state_dict()
    want = {"aabb": (2, 3)}
    for l, m in enumerate(_multires(levels)):
        r = [x * m for x in res[:3]] + [res[3]]
        for k, (a, b) in enumerate(COMBOS):
            want[f"grids.{l}.{k}"] = (1, C, r[b], r[a])       # scene/hexplane.py init_grid_param: [1, out, res_b, res_a]
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    for p in f._planes():
        assert p.stride(1) == 1 and p.is_contiguous(memory_format=torch.channels_last)


@pytest.mark.parametrize("bad", [dict(channels=16), dict(net_width=128), dict(multires=[1, 2, 4]), dict(defor_depth=2)])
def test_fused_field_still_refuses(bad):
    with pytest.raises(NotImplementedError):
        field.deform_network(_hyper(**bad))


def test_field_refuses_other_grids():
    for cfg, multires in ((_cfg(8), [1, 2]), (_cfg(64), [1, 2]), (_cfg(16), [1, 2, 4, 8, 16]), (_cfg(16), []),
                          (dict(_cfg(16), grid_dimensions=3), [1, 2])):
        with pytest.raises(NotImplementedError):
            field.HexPlaneField(1.6, cfg, multires)


def test_patch_hexplane_selects_by_configuration(capsys):
    from b200gs import launcher

    class Original:
        def __init__(self, bounds, planeconfig, multires):
            self.args = (bounds, planeconfig, multires)
            self.feat_dim = planeconfig["output_coordinate_dim"] * len(multires)

    mod = types.ModuleType("scene_deformation_standin")
    mod.HexPlaneField = Original
    assert launcher.patch_hexplane(mod) is mod
    factory = mod.HexPlaneField
    assert launcher.patch_hexplane(mod) is mod and mod.HexPlaneField is factory          # patching twice is a no-op
    for C, levels in ((16, 1), (16, 3), (32, 2), (32, 3), (16, 4)):
        g = mod.HexPlaneField(1.6, _cfg(C, (6, 5, 7, 9)), _multires(levels))
        assert isinstance(g, field.HexPlaneField) and g.feat_dim == C * levels
    capsys.readouterr()
    for cfg, multires in ((_cfg(8), [1, 2]), (_cfg(16), [1, 2, 4, 8, 16]), (dict(_cfg(16), grid_dimensions=3), [1, 2])):
        g = mod.HexPlaneField(1.6, cfg, multires)
        assert type(g) is Original and g.args == (1.6, cfg, multires)
        assert capsys.readouterr().err.count("\n") == 1


def _fake_desc(C, levels=2):
    d = _HexDesc()
    d.levels, d.channels = levels, C
    for l in range(levels):
        for a in range(4):
            d.res[l][a] = 8
        for k in range(6):
            d.plane[l][k] = 0x100000 + 0x10000 * (6 * l + k)
    d.aabb = 0x200000
    return d


def _calls(L, d, P):
    """Every entry point that takes a descriptor, with fake device pointers (nothing may be launched for a refused one)."""
    b, p = ctypes.byref(d), ctypes.c_longlong(P)
    return {
        "forward": lambda: L.b200gs_hexplane_forward(b, p, 0x300000, None, None, 0.5, 0x400000, None),
        "backward": lambda: L.b200gs_hexplane_backward(b, p, 0x300000, None, None, 0.5, 0x400000, 0x500000, None),
        "forward_masked": lambda: L.b200gs_hexplane_forward_masked(b, p, 0x300000, None, None, 0.5, 0x3F, None, 0x400000, None),
        "backward_masked": lambda: L.b200gs_hexplane_backward_masked(b, p, 0x300000, None, None, 0.5, 0x3F, None, None, 0x400000,
                                                                     0x500000, 0x600000, 1 << 20, None),
        "regulation": lambda: L.b200gs_hexplane_regulation(b, 0.1, 0.1, 0.1, 0x400000, None),
        "time_forward": lambda: L.b200gs_hexplane_time_forward(b, p, 0x300000, None, 0.5, 0x400000, 0x500000, 0, None),
        "time_backward": lambda: L.b200gs_hexplane_time_backward(b, p, 0x300000, None, 0.5, 0x400000, 0x500000, 0x600000,
                                                                 0x700000, 0x800000, 1 << 20, 0, None),
    }


def test_entry_points_refuse_channel_counts():
    L = _lib.lib()
    for C in (8, 64):
        d = _fake_desc(C)
        for name, call in _calls(L, d, 1000).items():
            assert call() != 0, (C, name)
            assert f"{C} channels".encode() in L.b200gs_last_error(), (C, name, L.b200gs_last_error())
        assert L.b200gs_hexplane_time_supported(ctypes.byref(d)) == 0
        assert L.b200gs_hexplane_time_row_scratch_bytes(ctypes.byref(d), 4) == 0
    d16 = _fake_desc(16)
    for name in ("time_forward", "time_backward"):          # the pre-blended time-row kernels are 32-channel only
        assert _calls(L, d16, 1000)[name]() != 0, name
        assert b"16 channels" in L.b200gs_last_error()
        assert _calls(L, d16, 0)[name]() != 0, name          # refused before anything else, empty launch or not
    assert L.b200gs_hexplane_time_supported(ctypes.byref(d16)) == 0
    # the six-plane entry points accept 16 channels (an empty launch validates the descriptor and returns)
    for name in ("forward", "backward", "forward_masked", "backward_masked"):
        assert _calls(L, d16, 0)[name]() == 0, (name, L.b200gs_last_error())
    # the row scratch is sized by the real channel count: (8 + 8 + 8) texels per level
    assert L.b200gs_hexplane_time_row_scratch_bytes(ctypes.byref(d16), 3) == 2 * 24 * 16 * 4 * 3
    assert L.b200gs_hexplane_time_row_scratch_bytes(ctypes.byref(_fake_desc(32)), 3) == 2 * 24 * 32 * 4 * 3


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against FP64
def _rel(a, b):
    return (a.double() - b.double()).abs().max().item() / max(b.abs().max().item(), 1e-30)


def _grid(C, levels, seed, res=(64, 48, 40, 150)):
    torch.manual_seed(seed)
    f = field.HexPlaneField(1.6, _cfg(C, res), _multires(levels)).cuda()
    with torch.no_grad():
        for p in f._planes():
            p.add_(torch.randn_like(p) * 0.1)
    f.set_aabb([1.0, 1.0, 1.0], [-1.0, -1.0, -1.0])
    return f


def _lattice(shape, g, lim=1.2):
    """Coordinates k / 1024: with the unit aabb of _grid the normalised coordinate and the pixel coordinate
    ((c + 1) / 2) (W - 1) are exact in FP32, so FP32 and FP64 pick the same texel for every point.  (A point within rounding
    distance of a texel edge would otherwise land in different cells, and its coordinate gradient, which jumps there, with it.)
    |c| up to `lim`: points outside the aabb exercise the border clamp."""
    k = int(lim * 1024)
    return torch.randint(-k, k + 1, shape, device="cuda", generator=g).float() / 1024


def _oracle(f, xyz, t, levels, dtype):
    """The reference's interpolate_ms_features (oracle restatement) in `dtype`, with leaf copies of every plane."""
    from oracle import field_torch
    planes = [p.detach().to(dtype).contiguous().requires_grad_(True) for p in f._planes()]
    x = xyz.detach().to(dtype).requires_grad_(True)
    feat = field_torch.hexplane_features(x, t.to(dtype).reshape(-1, 1), f.aabb.detach().to(dtype), planes, levels)
    return feat, x, planes


def _run_ours(f, xyz, times):
    for p in f._planes():
        p.grad = None
    x = xyz.clone().requires_grad_(True)
    feat = f(x, times)
    return feat, x


def _check_against_fp64(C, levels, P, uniform, seed):
    f = _grid(C, levels, seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    xyz = _lattice((P, 3), g)                                                     # some points outside the aabb: border clamp
    if uniform:
        t = torch.full((P, 1), 315 / 1024, device="cuda")                         # one timestamp: the row-reduced backward
    else:
        t = _lattice((P, 1), g)                                                   # per point, some outside [-1, 1]
    feat, x = _run_ours(f, xyz, t)
    assert feat.shape == (P, C * levels)
    w = torch.randn(P, C * levels, device="cuda", generator=g)
    (feat * w).sum().backward()
    ref, x64, planes64 = _oracle(f, xyz, t, levels, torch.float64)
    (ref * w.double()).sum().backward()
    assert _rel(feat, ref) <= 2e-6, (C, levels, P, _rel(feat, ref))
    assert _rel(x.grad, x64.grad) <= 1e-4, (C, levels, P, _rel(x.grad, x64.grad))
    for i, (p, q) in enumerate(zip(f._planes(), planes64)):
        assert _rel(p.grad, q.grad) <= 1e-4, (C, levels, P, i, _rel(p.grad, q.grad))
    return f, xyz, t, feat


CASES = [  # (P, levels, uniform time)
    (1, 1, False), (1, 2, True), (7, 2, False), (7, 4, True), (33, 3, True), (33, 1, False),
    (20000, 1, True), (20000, 2, False), (20000, 3, True), (20000, 4, False), (20000, 4, True),
    (1000003, 2, True), (1000003, 3, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("P,levels,uniform", CASES)
def test_sixteen_channels_against_fp64(P, levels, uniform):
    f16, xyz, t, feat16 = _check_against_fp64(16, levels, P, uniform, seed=11 + levels)
    # control: the 32-channel kernels on the same points, with the 16-channel planes as their first 16 channels.  A channel's
    # arithmetic does not depend on the layout, so those features agree bit for bit.
    f32 = _grid(32, levels, seed=11 + levels)
    with torch.no_grad():
        for p32, p16 in zip(f32._planes(), f16._planes()):
            p32[:, :16].copy_(p16)
    feat32, _ = _run_ours(f32, xyz, t)
    for l in range(levels):
        assert torch.equal(feat32[:, 32 * l: 32 * l + 16], feat16[:, 16 * l: 16 * (l + 1)]), l


@pytest.mark.gpu
@pytest.mark.parametrize("levels,uniform", [(2, True), (3, False)])
def test_thirty_two_channel_control_against_fp64(levels, uniform):
    _check_against_fp64(32, levels, 20000, uniform, seed=3)


@pytest.mark.gpu
@pytest.mark.parametrize("levels,T", [(1, 150), (2, 50), (3, 150), (4, 25)])
def test_regulation_sixteen_channels(levels, T):
    from oracle import field_torch
    f = _grid(16, levels, seed=7, res=(64, 48, 40, T))
    tw, l1w, pw = 0.01, 0.0001, 0.0001
    ref_grids = [[p.detach().clone().contiguous().requires_grad_(True) for p in gp] for gp in f.grids]
    ref = field_torch.plane_regulation(ref_grids, tw, l1w, pw)
    ref.backward()
    ours = field.compute_regulation(f, tw, l1w, pw)
    ours.backward()
    assert abs(ours.item() - ref.item()) < 1e-5 * abs(ref.item()), (ours.item(), ref.item())
    for p, q in zip(f._planes(), [q for rg in ref_grids for q in rg]):
        assert (p.grad - q.grad).abs().max().item() <= 1e-5 * q.grad.abs().max().item()
    before = [p.grad.clone() for p in f._planes()]
    acc = torch.zeros(1, device="cuda")
    field.accumulate_regulation(f, tw, l1w, pw, loss_accum=acc)
    assert abs(acc.item() - ref.item()) < 1e-5 * abs(ref.item())
    for p, b, q in zip(f._planes(), before, [q for rg in ref_grids for q in rg]):
        assert ((p.grad - b) - q.grad).abs().max().item() <= 1e-5 * q.grad.abs().max().item()


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the grid under the reference's own (PyTorch) MLP
@pytest.mark.gpu
def test_cell_order_of_per_call_copies():
    """The reference's Deformation hands the grid a fresh slice every call, so the grid sorts a fresh xyz copy every call
    (the freed copy's address, recycled for the next one, must not pass for the same points).  A long-lived contiguous
    tensor keeps its order until it changes."""
    P = 1 << 15
    f = _grid(16, 2, seed=41)
    g = torch.Generator(device="cuda").manual_seed(42)
    t = torch.full((P, 1), 0.25, device="cuda")
    c = _lib.COUNTERS
    with torch.no_grad():
        for _ in range(3):
            emb = torch.rand(P, 63, device="cuda", generator=g) * 2 - 1
            before = c["cell_order_sorts"]
            f(emb[:, :3], t)
            del emb                                  # its copy's memory is free for the next call
            assert c["cell_order_sorts"] == before + 1
        xyz = torch.rand(P, 3, device="cuda", generator=g) * 2 - 1
        f(xyz, t)
        before = c["cell_order_sorts"]
        a = f(xyz, t)
        assert c["cell_order_sorts"] == before
        xyz.copy_(xyz.flip(0))                       # an in-place change: the order is kept (a hint, ORDER_MAX_AGE versions)
        b = f(xyz, t)
        assert c["cell_order_sorts"] == before and torch.equal(b, a.flip(0))


@pytest.mark.gpu
def test_composed_field_under_reference_mlp():
    P, levels = 262144, 2
    f = _grid(16, levels, seed=21)
    torch.manual_seed(22)
    ours = StandInDeformation(f).cuda()
    ref64 = StandInDeformation(TorchGrid(f, torch.float64)).cuda().double().copy_mlp_from(ours)
    t32 = StandInDeformation(TorchGrid(f, torch.float32)).cuda().copy_mlp_from(ours)      # the reference as it runs: FP32
    g = torch.Generator(device="cuda").manual_seed(23)
    xyz = _lattice((P, 3), g, lim=1.0)
    # deform_network.forward_dynamic hands the grid a fresh [P, 63] positional encoding's first three columns
    emb = torch.cat([xyz, torch.randn(P, 60, device="cuda", generator=g)], 1)
    t = torch.full((P, 1), 431 / 1024, device="cuda")
    ws = [torch.randn(P, k, device="cuda", generator=g) for _, k in StandInDeformation.HEADS]

    def run(m, dtype):
        e = emb.detach().to(dtype).clone().requires_grad_(True)
        outs = m(e, t.to(dtype))
        sum((o * w.to(dtype)).sum() for o, w in zip(outs, ws)).backward()
        return outs, e.grad[:, :3]

    seen = {}

    def keep(mod, inp, out):                     # the grid's features and the upstream gradient the MLP hands back to it
        seen["feat"] = out
        out.register_hook(lambda gr: seen.__setitem__("d_feat", gr))
    hook = f.register_forward_hook(keep)
    o_ours, dx_ours = run(ours, torch.float32)
    hook.remove()
    # the grid alone, on exactly what it was given, at the flat grid bars
    from oracle import field_torch
    planes64 = [p.detach().double().contiguous().requires_grad_(True) for p in f._planes()]
    x64 = xyz.double().requires_grad_(True)
    feat64 = field_torch.hexplane_features(x64, t.double(), f.aabb.detach().double(), planes64, levels)
    feat64.backward(seen["d_feat"].double())
    assert _rel(seen["feat"], feat64) <= 2e-6
    assert _rel(dx_ours, x64.grad) <= 1e-4                  # xyz reaches the outputs through the grid only
    for i, (p, q) in enumerate(zip(f._planes(), planes64)):
        assert _rel(p.grad, q.grad) <= 1e-4, (i, _rel(p.grad, q.grad))
    # the whole field against the same module in FP64
    o_64, dx_64 = run(ref64, torch.float64)
    o_32, dx_32 = run(t32, torch.float32)

    def err(a, ref):
        return ((a.double() - ref).abs().max() / ref.abs().max()).item()

    for a, b, r in zip(o_ours, o_32, o_64):
        assert err(a, r) <= max(1e-5, 2 * err(b, r)), (err(a, r), err(b, r))
    assert err(dx_ours, dx_64) <= max(1e-3, 2 * err(dx_32, dx_64))
    named64, named32 = dict(ref64.named_parameters()), dict(t32.named_parameters())
    checked = 0
    for n, p in ours.named_parameters():
        if not p.requires_grad:                  # grid.aabb
            continue
        if n.startswith("grid."):
            # End to end, a plane's gradient carries the MLP's error: at this size a few hidden pre-activations sit within FP32
            # rounding of 0, their ReLU masks differ from FP64's and so does d_features (FP32 PyTorch: a few 1e-3).  The grid's
            # own share is held to the flat 1e-4 above; here it is anchored like the MLP.
            l, j = (int(x) for x in n.split(".")[-2:])            # grid.grids.{level}.{plane}
            n64, bar = f"grid.planes.{6 * l + j}", 1e-4
        else:                                    # the MLP: anchored on FP32 PyTorch (DESIGN.md section 5)
            n64, bar = n, 1e-3
        e_ours, e_t32 = err(p.grad, named64[n64].grad), err(named32[n64].grad, named64[n64].grad)
        assert e_ours <= max(bar, 2 * e_t32), (n, e_ours, e_t32)
        checked += 1
    assert checked == 6 * levels + 2 + 4 * 5


@pytest.mark.gpu
def test_fused_adam_step_on_sixteen_channel_planes():
    from b200gs.adam import FusedAdam
    f_a, f_b = _grid(16, 3, seed=31), _grid(16, 3, seed=31)
    g = torch.Generator(device="cuda").manual_seed(32)
    for pa, pb in zip(f_a._planes(), f_b._planes()):
        gr = (torch.randn(pa.shape, device="cuda", generator=g) * 1e-3).contiguous(memory_format=torch.channels_last)
        pa.grad, pb.grad = gr.clone(memory_format=torch.preserve_format), gr.clone(memory_format=torch.preserve_format)
    ref = torch.optim.Adam([{"params": f_a._planes(), "lr": 1.6e-3, "name": "grid"}], lr=0.0, eps=1e-15)
    ours = FusedAdam([{"params": f_b._planes(), "lr": 1.6e-3, "name": "grid"}], lr=0.0, eps=1e-15)
    ref.step(); ours.step()
    for pa, pb in zip(f_a._planes(), f_b._planes()):
        assert pb.stride() == pa.stride() and pb.stride(1) == 1
        assert torch.equal(pa.detach(), pb.detach())
        assert torch.equal(ref.state[pa]["exp_avg"], ours.state[pb]["exp_avg"])
        assert torch.equal(ref.state[pa]["exp_avg_sq"], ours.state[pb]["exp_avg_sq"])
