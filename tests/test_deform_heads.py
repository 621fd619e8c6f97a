"""The opacity and SH deformation heads (no_do = False, no_dshs = False; csrc/deform_heads.cu, include/b200gs.h
b200gs_deform_heads_*): their plain-PyTorch restatement, the parameter set the trainer's arena covers, argument validation, the
kernels against FP64, the field module against that restatement, the trainer's fast path against plain autograd, and rendering.

Kernel metric (as tests/test_deform_mlp_kernels.py): |y - y64| <= eps * M, M = the same FP64 chain on |W|, |b| and
|activations| under the FP64 ReLU masks; inputs keep a ReLU margin so that the masks of FP64 and the kernels agree.
  outputs, d_features        2^-17   three-term TF32 split, FP32 accumulation
  weight / bias gradients    2^-9    against FP64 (X rounded to TF32 once)
                             2^-16   against the modelled rounding (P >= 1024): dY exact, X = the stashed FP32 activation or
                                     the feature rounded with cvt.rna (dW1, dW2 and dW3 alike), bias gradients exact sums.
"""
import copy
import ctypes
import math
import os
import sys
import types

import pytest
import torch
import torch.nn.functional as Fn

from b200gs import _lib
from b200gs.field import _HeadsGrads, _HeadsWeights, _MlpWeights
from oracle import field_torch as oracle

MW = 64
KD = (1, 48)
EPS_FWD = 2.0 ** -17
EPS_W64 = 2.0 ** -9
EPS_WMOD = 2.0 ** -16
MODELLED_MIN_P = 1024
SENTINEL = -12345.5
REF = "/root/reference"
HEAD_MASKS = {"op": (True, False), "sh": (False, True), "op+sh": (True, True)}


def tf32_rna(x):
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def stash_index(P, cols=MW):
    r = torch.arange(P, dtype=torch.int64)[:, None]
    c = torch.arange(cols, dtype=torch.int64)[None, :]
    return (r >> 7) * (128 * MW) + ((r & 127) >> 2) * 256 + (c >> 2) * 16 + (r & 3) * 4 + (c & 3)


def stash_plane_floats(P):
    return (P + 127) // 128 * 128 * MW


def ratio(y, ref, M, eps):
    d = (y.to(torch.float64) - ref.to(torch.float64)).abs()
    lim = eps * M.to(torch.float64)
    r = torch.where(lim > 0, d / torch.where(lim > 0, lim, 1.0), torch.where(d > 0, math.inf, 0.0))
    r = torch.where(torch.isfinite(d), r, math.inf)
    return r.max().item() if r.numel() else 0.0


# ---------------------------------------------------------------------------------------------------------------------------
# the reference's field with the opacity / SH heads, in plain PyTorch
def deform_forward(sd, levels, point, scales, rotations, opacity, shs, times_sel, scene_flow, frame_num, delta_scale,
                   no_do=True, no_dshs=True):
    """oracle.field_torch.deform_forward (HexPlane features, hidden, the three geometry heads) plus the opacity and SH heads
    of scene/deformation.py:97-153 with mask = ones, restated operator for operator:
        opacity' = opacity[:, :1] * mask + opacity_deform(hidden);  shs' = shs * mask[..., None] + shs_deform(hidden).reshape(P,16,3)
    With both flags True it is oracle.field_torch.deform_forward itself."""
    pts, sc, rt, op, sh = oracle.deform_forward(sd, levels, point, scales, rotations, opacity, shs, times_sel, scene_flow,
                                                frame_num, delta_scale)
    if no_do and no_dshs:
        return pts, sc, rt, op, sh
    planes = [sd[f"deformation_net.grid.grids.{l}.{k}"] for l in range(levels) for k in range(6)]
    feat = oracle.hexplane_features(point[:, :3], times_sel[:, :1], sd["deformation_net.grid.aabb"], planes, levels)
    hidden = Fn.linear(feat, sd["deformation_net.feature_out.0.weight"], sd["deformation_net.feature_out.0.bias"])
    mask = torch.ones_like(opacity[:, 0]).unsqueeze(-1)

    def head(name):
        x = Fn.linear(torch.relu(hidden), sd[f"deformation_net.{name}.1.weight"], sd[f"deformation_net.{name}.1.bias"])
        return Fn.linear(torch.relu(x), sd[f"deformation_net.{name}.3.weight"], sd[f"deformation_net.{name}.3.bias"])
    if not no_do:
        op = opacity[:, :1] * mask + head("opacity_deform")
    if not no_dshs:
        sh = shs * mask.unsqueeze(-1) + head("shs_deform").reshape([shs.shape[0], 16, 3])
    return pts, sc, rt, op, sh


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: the restatement, arena, refusals
def _hyper(no_do=False, no_dshs=False, width=64, channels=32):
    return types.SimpleNamespace(
        net_width=width, timebase_pe=4, defor_depth=0, posebase_pe=10, scale_rotation_pe=2, opacity_pe=2,
        timenet_width=64, timenet_output=32, bounds=1.6, grid_pe=0, plane_tv_weight=0.0001, time_smoothness_weight=0.01,
        l1_time_planes=0.0001,
        kplanes_config={'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': channels,
                        'resolution': [64, 64, 64, 50]},
        multires=[1, 2], no_dx=False, no_grid=False, no_ds=False, no_dr=False, no_do=no_do, no_dshs=no_dshs,
        empty_voxel=False, static_mlp=False, apply_rotation=False)


def _state_dict(levels, seed, dtype=torch.float64, res=(8, 8, 8, 5)):
    g = torch.Generator().manual_seed(seed)
    sd = {"deformation_net.grid.aabb": torch.tensor([[1.6] * 3, [-1.6] * 3], dtype=dtype)}
    combos = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    for l in range(levels):
        for k, (a, b) in enumerate(combos):
            sd[f"deformation_net.grid.grids.{l}.{k}"] = (torch.rand(1, 32, res[b], res[a], generator=g) + 0.5).to(dtype)
    lin = lambda o, i: ((torch.rand(o, i, generator=g) * 2 - 1) / math.sqrt(i), torch.randn(o, generator=g) * 0.1)
    sd["deformation_net.feature_out.0.weight"], sd["deformation_net.feature_out.0.bias"] = lin(64, 32 * levels)
    for name, k in (("pos_deform", 3), ("scales_deform", 3), ("rotations_deform", 4), ("opacity_deform", 1), ("shs_deform", 48)):
        sd[f"deformation_net.{name}.1.weight"], sd[f"deformation_net.{name}.1.bias"] = lin(64, 64)
        sd[f"deformation_net.{name}.3.weight"], sd[f"deformation_net.{name}.3.bias"] = lin(k, 64)
    return {k: v.to(dtype).requires_grad_(True) for k, v in sd.items()}


@pytest.mark.parametrize("no_do,no_dshs", [(False, True), (True, False), (False, False)])
def test_restatement_heads_match_fp64_formulas(no_do, no_dshs):
    """The restatement's opacity / SH branches against an independent FP64 statement of deformation.py:97-153 (mask = ones),
    values and autograd gradients of every input and head parameter."""
    P, levels = 300, 2
    g = torch.Generator().manual_seed(4)
    d = torch.float64
    sd = _state_dict(levels, 5)
    xyz = (torch.rand(P, 3, generator=g, dtype=d) * 3 - 1.5)
    scales, rot = torch.randn(P, 3, generator=g, dtype=d), torch.randn(P, 4, generator=g, dtype=d)
    opacity = torch.randn(P, 1, generator=g, dtype=d).requires_grad_(True)
    shs = torch.randn(P, 16, 3, generator=g, dtype=d).requires_grad_(True)
    t = torch.rand(P, 1, generator=g, dtype=d)
    flow = torch.randn(P, 3, generator=g, dtype=d)
    _, _, _, op, sh = deform_forward(sd, levels, xyz, scales, rot, opacity, shs, t, flow, 3.0, 0.5, no_do=no_do, no_dshs=no_dshs)
    planes = [sd[f"deformation_net.grid.grids.{l}.{k}"] for l in range(levels) for k in range(6)]
    feat = oracle.hexplane_features(xyz, t, sd["deformation_net.grid.aabb"], planes, levels)
    hidden = feat @ sd["deformation_net.feature_out.0.weight"].T + sd["deformation_net.feature_out.0.bias"]

    def head(name):
        z = torch.relu(torch.relu(hidden) @ sd[f"deformation_net.{name}.1.weight"].T + sd[f"deformation_net.{name}.1.bias"])
        return z @ sd[f"deformation_net.{name}.3.weight"].T + sd[f"deformation_net.{name}.3.bias"]
    op_ref = opacity if no_do else opacity + head("opacity_deform")
    sh_ref = shs if no_dshs else shs + head("shs_deform").reshape(P, 16, 3)
    assert torch.allclose(op, op_ref, rtol=1e-12, atol=1e-12) and torch.allclose(sh, sh_ref, rtol=1e-12, atol=1e-12)
    wo, ws = torch.randn(P, 1, generator=g, dtype=d), torch.randn(P, 16, 3, generator=g, dtype=d)
    names = [k for k in sd if ("opacity_deform" in k and not no_do) or ("shs_deform" in k and not no_dshs) or "feature_out" in k]
    tensors = [opacity, shs] + [sd[k] for k in names]
    ga = torch.autograd.grad((op * wo).sum() + (sh * ws).sum(), tensors, allow_unused=True)
    gb = torch.autograd.grad((op_ref * wo).sum() + (sh_ref * ws).sum(), tensors, allow_unused=True)
    for n, a, b in zip(["opacity", "shs"] + names, ga, gb):
        assert (a is None) == (b is None), n
        if a is not None:
            assert torch.allclose(a, b, rtol=1e-10, atol=1e-12), n
    assert all(x is not None for x in ga[2:]), "every parameter of an enabled head (and feature_out) receives a gradient"


def test_restatement_without_heads_is_the_oracle():
    sd = _state_dict(2, 6)
    g = torch.Generator().manual_seed(1)
    P = 50
    args = [torch.rand(P, 3, generator=g, dtype=torch.float64), torch.randn(P, 3, generator=g, dtype=torch.float64),
            torch.randn(P, 4, generator=g, dtype=torch.float64), torch.randn(P, 1, generator=g, dtype=torch.float64),
            torch.randn(P, 16, 3, generator=g, dtype=torch.float64), torch.rand(P, 1, generator=g, dtype=torch.float64),
            torch.randn(P, 3, generator=g, dtype=torch.float64)]
    out = deform_forward(sd, 2, *args, 2.0, 1.0)
    ref = oracle.deform_forward(sd, 2, *args, 2.0, 1.0)
    assert all(torch.equal(a, b) for a, b in zip(out, ref))
    assert torch.equal(out[3], args[3][:, :1]) and out[4] is args[4]


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "scene")), reason="reference tree not present")
def test_restatement_heads_match_reference_module():
    """With both flags off the restatement equals the reference's own Deformation (scene/deformation.py) on the same weights."""
    saved_path, saved_mods = list(sys.path), set(sys.modules)
    try:
        sys.path.insert(0, REF)
        from scene.deformation import deform_network as ref_net
        torch.manual_seed(0)
        h = _hyper()
        h.kplanes_config = dict(h.kplanes_config, resolution=[8, 8, 8, 5])
        net = ref_net(h)
        sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
        P = 200
        g = torch.Generator().manual_seed(2)
        xyz, sc, rt = torch.rand(P, 3, generator=g) * 2 - 1, torch.randn(P, 3, generator=g), torch.randn(P, 4, generator=g)
        op, shs, t = torch.randn(P, 1, generator=g), torch.randn(P, 16, 3, generator=g), torch.rand(P, 1, generator=g)
        flow = torch.zeros(P, 3)
        with torch.no_grad():
            r = net(xyz, sc, rt, op, shs, t, flow, torch.tensor(0.0), 1.0)
            o = deform_forward(sd, 2, xyz, sc, rt, op, shs, t, flow, 0.0, 1.0, no_do=False, no_dshs=False)
        for a, b in zip(r, o):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)
    finally:
        sys.path[:] = saved_path
        for m in set(sys.modules) - saved_mods:
            sys.modules.pop(m, None)


def test_receives_grad_adds_exactly_the_enabled_heads():
    from b200gs import engine
    from b200gs.field import deform_network
    names = [n for n, _ in deform_network(_hyper()).named_parameters()]
    names = ["_deformation." + n for n in names] + ["_xyz", "_features_dc", "_opacity"]
    old = lambda n: not n.startswith("_deformation.") or not ("timenet" in n or "opacity_deform" in n or "shs_deform" in n
                                                              or n.endswith("grid.aabb"))
    base = {n for n in names if engine._receives_grad(n, "fine")}
    assert base == {n for n in names if old(n)}
    assert base == {n for n in names if engine._receives_grad(n, "fine", no_do=True, no_dshs=True)}
    for no_do, no_dshs, tag in ((False, True, "opacity_deform"), (True, False, "shs_deform")):
        s = {n for n in names if engine._receives_grad(n, "fine", no_do, no_dshs)}
        assert s - base == {n for n in names if tag in n} and len(s - base) == 4 and base <= s
    both = {n for n in names if engine._receives_grad(n, "fine", False, False)}
    assert both - base == {n for n in names if "opacity_deform" in n or "shs_deform" in n}
    assert not any(engine._receives_grad(n, "coarse", False, False) for n in names if n.startswith("_deformation."))


def test_field_accepts_heads_and_still_refuses_the_rest():
    from b200gs.field import deform_network
    for no_do, no_dshs in ((False, True), (True, False), (False, False)):
        deform_network(_hyper(no_do, no_dshs))
    for bad in (dict(width=128), dict(channels=16)):
        with pytest.raises(NotImplementedError):
            deform_network(_hyper(**bad))
    h = _hyper()
    h.defor_depth = 2
    with pytest.raises(NotImplementedError):
        deform_network(h)


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference tree not present")
def test_launcher_builds_fused_field_with_heads():
    saved_path, saved_mods = list(sys.path), set(sys.modules)
    try:
        from b200gs import launcher
        gm = launcher.install(REF)
        h = _hyper(no_do=False)
        h.kplanes_config = dict(h.kplanes_config, resolution=[8, 8, 8, 5])
        assert type(gm.GaussianModel(3, h)._deformation).__module__ == "b200gs.field"
        wide = copy.deepcopy(h); wide.net_width = 128
        wide.kplanes_config = dict(h.kplanes_config, output_coordinate_dim=16)
        assert type(gm.GaussianModel(3, wide)._deformation).__module__ == "scene.deformation"
    finally:
        sys.path[:] = saved_path
        for m in set(sys.modules) - saved_mods:
            sys.modules.pop(m, None)


def _fake_hw(F=64, width=MW, tiled=0, heads=(True, True)):
    w = _HeadsWeights(feat_dim=F, width=width, w1=0x10000, feat_tiled=tiled)
    for h in range(2):
        if heads[h]:
            w.w2[h], w.b2[h], w.w3[h], w.b3[h] = 0x30000 + 0x1000 * h, 0x40000 + 0x1000 * h, 0x50000 + 0x1000 * h, 0x60000 + 0x1000 * h
    return w


def _fake_hg(**over):
    gw = _HeadsGrads(w1=0x70000, b1=0x80000)
    for h in range(2):
        gw.w2[h], gw.b2[h], gw.w3[h], gw.b3[h] = 0x90000 + 0x1000 * h, 0xa0000 + 0x1000 * h, 0xb0000 + 0x1000 * h, 0xc0000 + 0x1000 * h
    for k, v in over.items():
        if "_" in k:
            name, h = k.split("_")
            getattr(gw, name)[int(h)] = v
        else:
            setattr(gw, k, v)
    return gw


def _hfwd(L, w, P, sh=16):
    return L.b200gs_deform_heads_forward(ctypes.byref(w), ctypes.c_longlong(P), sh, 0xd0000, 0xe0000, 0xe1000, 0xe2000, 0xe3000,
                                         0xe4000, None)


def _hbwd(L, w, P, sh=16, gw=None):
    return L.b200gs_deform_heads_backward(ctypes.byref(w), ctypes.byref(gw or _fake_hg()), ctypes.c_longlong(P), sh, 0xe0000,
                                          0xd0000, 0xd8000, 0xe1000, 0xe2000, 0xe3000, 0xe4000, 0, None)


def test_heads_entry_points_refuse_bad_arguments():
    """Each refusal comes back with a message before anything is launched (the fake device pointers would fault)."""
    L = _lib.lib()
    for what, w, sh in (("SH coefficients", _fake_hw(), 9), ("net_width", _fake_hw(width=128), 16),
                        ("feature dim", _fake_hw(F=96), 16), ("both heads are off", _fake_hw(heads=(False, False)), 16)):
        for call in (_hfwd, _hbwd):
            assert call(L, w, 1000, sh) != 0, (what, call.__name__)
            assert what.encode() in L.b200gs_last_error(), (what, L.b200gs_last_error())
    # the SH count only matters with the SH head on
    for what, gw in (("dW1", _fake_hg(w1=0x70004)), ("head 0 weight gradient not 16-byte aligned", _fake_hg(w2_0=0x90008)),
                     ("head 1 weight gradient not 16-byte aligned", _fake_hg(w3_1=0xb1004))):
        assert _hbwd(L, _fake_hw(), 1000, gw=gw) != 0
        assert what.encode() in L.b200gs_last_error(), (what, L.b200gs_last_error())
    for P in (0, -1):                      # empty launches return before touching anything
        assert _hfwd(L, _fake_hw(), P) == 0 and _hbwd(L, _fake_hw(), P) == 0
        assert _hfwd(L, _fake_hw(heads=(True, False)), P, sh=9) == 0
    assert L.b200gs_deform_heads_saved_floats(0) == 0
    assert L.b200gs_deform_heads_saved_floats(129) == 2 * 256 * MW


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against FP64
def _weights(F, seed):
    g = torch.Generator().manual_seed(seed)

    def lin(o, i):
        bd = 1.0 / math.sqrt(i)
        return ((torch.rand(o, i, generator=g) * 2 - 1) * bd,
                (torch.rand(o, generator=g) * 2 - 1) * bd + torch.randn(o, generator=g) * 0.05)
    W = {}
    W["w1"], W["b1"] = lin(MW, F)
    for h in range(3):                      # the three geometry heads (their forward leaves the stash)
        W[f"g2_{h}"], W[f"gb2_{h}"] = lin(MW, MW)
        W[f"g3_{h}"], W[f"gb3_{h}"] = lin((3, 3, 4)[h], MW)
    for h in range(2):
        W[f"w2_{h}"], W[f"b2_{h}"] = lin(MW, MW)
        W[f"w3_{h}"], W[f"b3_{h}"] = lin(KD[h], MW)
    return W


GRADS = ("w1", "b1", "w2_0", "b2_0", "w3_0", "b3_0", "w2_1", "b2_1", "w3_1", "b3_1")


def _draw(F, P, W, seed, dev):
    """Feature rows whose hidden and heads' layer-2 pre-activations keep a ReLU margin, plus inputs and upstream gradients."""
    g = torch.Generator(device=dev).manual_seed(seed)
    Wd = {k: v.to(dev, torch.float64) for k, v in W.items()}
    kept, n_kept = [], 0
    while n_kept < P:
        n = int(1.3 * (P - n_kept)) + 16
        feat = torch.randn(n, F, generator=g, device=dev) * 0.6 + 0.15
        fd = feat.double()
        a1 = fd @ Wd["w1"].T + Wd["b1"]
        A1 = fd.abs() @ Wd["w1"].abs().T + Wd["b1"].abs()
        ok = (a1.abs() >= 1e-4 * A1.mean()).all(1)
        hdn, Mh = a1.clamp_min(0), A1 * (a1 > 0)
        for h in range(2):
            a2 = hdn @ Wd[f"w2_{h}"].T + Wd[f"b2_{h}"]
            ok &= (a2.abs() >= 1e-4 * (Mh @ Wd[f"w2_{h}"].abs().T + Wd[f"b2_{h}"].abs()).mean()).all(1)
        kept.append(feat[ok])
        n_kept += int(ok.sum())
    x = {"feat": torch.cat(kept)[:P].contiguous(),
         "op": torch.randn(P, 1, generator=g, device=dev) * 2,
         "shs": torch.randn(P, 48, generator=g, device=dev),
         "dop": torch.randn(P, 1, generator=g, device=dev) + 0.5,
         "dsh": torch.randn(P, 48, generator=g, device=dev) + 0.5}
    return x


def _reference(W, x, on, dev):
    """FP64 outputs, gradients (incl. dz, dh for the model) and magnitudes M."""
    d = torch.float64
    Wd = {k: v.to(dev, d) for k, v in W.items()}
    feat = x["feat"].double()
    a1 = feat @ Wd["w1"].T + Wd["b1"]
    m1 = (a1 > 0).double()
    hdn = a1 * m1
    Mh = (feat.abs() @ Wd["w1"].abs().T + Wd["b1"].abs()) * m1
    ref, M = {}, {}
    drh, Mdrh = torch.zeros_like(a1), torch.zeros_like(a1)
    for h in range(2):
        if not on[h]:
            continue
        base, dout = (x["op"], x["dop"]) if h == 0 else (x["shs"], x["dsh"])
        base, dout = base.double(), dout.double()
        w2, b2, w3, b3 = (Wd[f"{n}_{h}"] for n in ("w2", "b2", "w3", "b3"))
        a2 = hdn @ w2.T + b2
        m2 = (a2 > 0).double()
        z = a2 * m2
        Mz = (Mh @ w2.abs().T + b2.abs()) * m2
        ref[f"out_{h}"] = base + (z @ w3.T + b3)
        M[f"out_{h}"] = base.abs() + Mz @ w3.abs().T + b3.abs()
        dz = (dout @ w3) * m2
        Mdz = (dout.abs() @ w3.abs()) * m2
        drh, Mdrh = drh + dz @ w2, Mdrh + Mdz @ w2.abs()
        ref[f"w3_{h}"], M[f"w3_{h}"] = dout.T @ z, dout.abs().T @ Mz
        ref[f"b3_{h}"], M[f"b3_{h}"] = dout.sum(0), dout.abs().sum(0)
        ref[f"w2_{h}"], M[f"w2_{h}"] = dz.T @ hdn, Mdz.T @ Mh
        ref[f"b2_{h}"], M[f"b2_{h}"] = dz.sum(0), Mdz.sum(0)
        ref[f"dz_{h}"] = dz
    dh, Mdh = drh * m1, Mdrh * m1
    ref["dh"] = dh
    ref["dfeat"], M["dfeat"] = dh @ Wd["w1"], Mdh @ Wd["w1"].abs()
    ref["w1"], M["w1"] = dh.T @ feat, Mdh.T @ feat.abs()
    ref["b1"], M["b1"] = dh.sum(0), Mdh.sum(0)
    return ref, M


def _run(F, tiled, on, P, W, x, dev, *, M_dfeat=None, sh_overwrite=0, heads_stash=True, seed=0):
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    nan = float("nan")
    Wd = {k: v.to(dev).contiguous() for k, v in W.items()}
    n_tiles = (P + 127) // 128
    idx = stash_index(P).to(dev)
    if tiled:
        fbuf = torch.full(((n_tiles + 1) * 128 * MW,), nan, device=dev)
        fbuf[idx] = x["feat"]
    else:
        fbuf = torch.full((P + 3, F), nan, device=dev)
        fbuf[:P] = x["feat"]
    # the three-head forward leaves relu(hidden) in plane 0 of its stash
    n_saved = L.b200gs_deform_mlp_saved_floats(P)
    saved = torch.full((n_saved,), nan, device=dev)
    mw = _MlpWeights(feat_dim=F, width=MW, w1=Wd["w1"].data_ptr(), b1=Wd["b1"].data_ptr(), feat_tiled=int(tiled))
    for h in range(3):
        mw.w2[h], mw.b2[h], mw.w3[h], mw.b3[h] = (Wd[f"{n}_{h}"].data_ptr() for n in ("g2", "gb2", "g3", "gb3"))
    geo = [torch.zeros(P, k, device=dev) for k in (3, 3, 4, 3)]
    geo_out = [torch.empty(P, k, device=dev) for k in (3, 3, 4)]
    assert L.b200gs_deform_mlp_forward(ctypes.byref(mw), P, fbuf.data_ptr(), *[t.data_ptr() for t in geo], 0.0, None, 0.0,
                                       *[t.data_ptr() for t in geo_out], saved.data_ptr(), stream) == 0, L.b200gs_last_error()

    hw = _HeadsWeights(feat_dim=F, width=MW, w1=Wd["w1"].data_ptr(), feat_tiled=int(tiled))
    for h in range(2):
        if on[h]:
            hw.w2[h], hw.b2[h], hw.w3[h], hw.b3[h] = (Wd[f"{n}_{h}"].data_ptr() for n in ("w2", "b2", "w3", "b3"))
    outs = [torch.full((P + 2, k), SENTINEL, device=dev) for k in KD]
    ins = [torch.cat((x[k], torch.full((2, x[k].shape[1]), nan, device=dev))) for k in ("op", "shs")]
    n_h = L.b200gs_deform_heads_saved_floats(P)
    assert n_h == 2 * stash_plane_floats(P)
    hs = torch.full((n_h + 64,), nan, device=dev)
    hs[n_h:] = SENTINEL
    rc = L.b200gs_deform_heads_forward(ctypes.byref(hw), P, 16, saved.data_ptr(), ins[0].data_ptr(), ins[1].data_ptr(),
                                       outs[0].data_ptr(), outs[1].data_ptr(), hs.data_ptr() if heads_stash else None, stream)
    assert rc == 0, L.b200gs_last_error()
    torch.cuda.synchronize()
    r = types.SimpleNamespace()
    for h in range(2):
        if on[h]:
            assert bool((outs[h][P:] == SENTINEL).all()), "forward wrote past row P"
        else:
            assert bool((outs[h] == SENTINEL).all()), f"disabled head {h} wrote its output"
    r.out = [o[:P].clone() for o in outs]
    assert bool((hs[n_h:] == SENTINEL).all()), "forward wrote past b200gs_deform_heads_saved_floats(P)"
    r.stash_h = saved[idx].clone()
    r.stash_z = [hs[h * stash_plane_floats(P) + idx].clone() for h in range(2)]
    if not heads_stash:
        return r

    # backward into pre-filled buffers
    g = torch.Generator(device=dev).manual_seed(seed)
    # d_features pre-filled at 1/16 of each element's magnitude M: adding instead of writing is then visible far above the
    # bound, while the FP32 rounding of the sum stays at the scale of the heads' share (a point whose few upstream gradients
    # are all near 0 has a tiny M; a fixed-size fill would round away more than its whole share)
    G = (M_dfeat.float() * (torch.rand(P, F, generator=g, device=dev) + 0.5) / 16 *
         torch.sign(torch.randn(P, F, generator=g, device=dev)))
    if tiled:
        dfeat = torch.full(((n_tiles + 1) * 128 * MW,), SENTINEL, device=dev)
        dfeat[idx] = G
    else:
        dfeat = torch.full((P + 3, F), SENTINEL, device=dev)
        dfeat[:P] = G
    r.G = G
    r.G0, bufs = {}, {}
    hg = _HeadsGrads()
    shapes = {"w1": (MW, F), "b1": (MW,)}
    for h in range(2):
        shapes.update({f"w2_{h}": (MW, MW), f"b2_{h}": (MW,), f"w3_{h}": (KD[h], MW), f"b3_{h}": (KD[h],)})
    for name, shp in shapes.items():
        n = math.prod(shp)
        r.G0[name] = (torch.randn(shp, generator=g, device=dev) * 0.01).cpu()
        buf = torch.full((n + 8,), SENTINEL, device=dev)
        buf[:n] = r.G0[name].reshape(-1).to(dev)
        bufs[name] = buf
        if "_" in name:
            getattr(hg, name.split("_")[0])[int(name[-1])] = buf.data_ptr()
        else:
            setattr(hg, name, buf.data_ptr())
    douts = [torch.cat((x[k], torch.full((2, x[k].shape[1]), nan, device=dev))) for k in ("dop", "dsh")]
    S0 = torch.randn(P, 48, generator=g, device=dev)
    shg = torch.full((P + 2, 48), SENTINEL, device=dev)
    shg[:P] = S0
    rc = L.b200gs_deform_heads_backward(ctypes.byref(hw), ctypes.byref(hg), P, 16, fbuf.data_ptr(), saved.data_ptr(),
                                        hs.data_ptr(), douts[0].data_ptr(), douts[1].data_ptr(), dfeat.data_ptr(),
                                        shg.data_ptr(), sh_overwrite, stream)
    assert rc == 0, L.b200gs_last_error()
    torch.cuda.synchronize()
    if tiled:
        r.dfeat = dfeat[idx].clone()
        rest = torch.ones_like(dfeat, dtype=torch.bool)
        rest[idx] = False
        assert bool((dfeat[rest] == SENTINEL).all()), "backward wrote a tiled d_features slot past row P"
    else:
        r.dfeat = dfeat[:P].clone()
        assert bool((dfeat[P:] == SENTINEL).all()), "backward wrote d_features past row P"
    assert bool((shg[P:] == SENTINEL).all()), "backward wrote the SH gradient past row P"
    if on[1]:
        want = x["dsh"] if sh_overwrite else S0 + x["dsh"]
        assert torch.equal(shg[:P], want), "SH gradient buffer != d shs' (written) / + d shs' (added)"
    else:
        assert torch.equal(shg[:P], S0), "the SH gradient buffer was touched with the SH head off"
    r.gw = {}
    for name, buf in bufs.items():
        n = math.prod(shapes[name])
        assert bool((buf[n:] == SENTINEL).all()), f"backward wrote past the end of the {name} gradient"
        if "_" in name and not on[int(name[-1])]:
            assert torch.equal(buf[:n].cpu(), r.G0[name].reshape(-1)), f"gradient of disabled head ({name}) was touched"
            continue
        r.gw[name] = buf[:n].reshape(shapes[name]).cpu()
    return r


def _check(F, on, P, r, ref, M, x, label):
    worst = {}
    for h in range(2):
        if on[h]:
            worst[f"out_{h}"] = ratio(r.out[h], ref[f"out_{h}"], M[f"out_{h}"], EPS_FWD)
    worst["dfeat"] = ratio(r.dfeat.double() - r.G.double(), ref["dfeat"], M["dfeat"], EPS_FWD)
    d64 = {k: v.double() - r.G0[k].double() for k, v in r.gw.items()}
    cpu = lambda t: t.cpu()
    for k, v in d64.items():
        worst["fp64:" + k] = ratio(v, cpu(ref[k]), cpu(M[k]), EPS_W64)
    if P >= MODELLED_MIN_P:
        d = torch.float64
        mod = {"w1": ref["dh"].T @ tf32_rna(x["feat"]).to(d), "b1": ref["b1"]}
        for h in range(2):
            if on[h]:
                dout = (x["dop"], x["dsh"])[h].to(d)
                mod[f"w3_{h}"] = dout.T @ tf32_rna(r.stash_z[h]).to(d)
                mod[f"w2_{h}"] = ref[f"dz_{h}"].T @ tf32_rna(r.stash_h).to(d)
                mod[f"b3_{h}"], mod[f"b2_{h}"] = ref[f"b3_{h}"], ref[f"b2_{h}"]
        for k, v in d64.items():
            worst["mod:" + k] = ratio(v, cpu(mod[k]), cpu(M[k]), EPS_WMOD)
    print(f"[deform-heads F={F} {label} P={P}] " + " ".join(f"{k}={v:.3g}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad


LAYOUTS = ((64, False), (64, True), (128, False))
KERNEL_P = (1, 127, 128, 129, 5000, 1000003)


@pytest.mark.gpu
@pytest.mark.parametrize("F,tiled", LAYOUTS, ids=("F64", "F64tiled", "F128"))
@pytest.mark.parametrize("heads", list(HEAD_MASKS))
@pytest.mark.parametrize("P", KERNEL_P)
def test_deform_heads_match_fp64(F, tiled, heads, P):
    dev = torch.device("cuda")
    on = HEAD_MASKS[heads]
    W = _weights(F, 200 + F)
    x = _draw(F, P, W, 7 * P + F, dev)
    ref, M = _reference(W, x, on, dev)
    r = _run(F, tiled, on, P, W, x, dev, M_dfeat=M["dfeat"], sh_overwrite=P % 2, seed=P)
    _check(F, on, P, r, ref, M, x, heads)
    if P == 5000:
        # inference (no heads stash) gives the same bits
        r2 = _run(F, tiled, on, P, W, x, dev, heads_stash=False)
        for h in range(2):
            assert torch.equal(r2.out[h], r.out[h])


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the field module against the restatement
def _model(no_do, no_dshs, seed=0):
    from b200gs.field import deform_network
    torch.manual_seed(seed)
    net = deform_network(_hyper(no_do, no_dshs)).cuda()
    with torch.no_grad():
        for p in net.deformation_net.grid.grids.parameters():
            p.add_(torch.randn_like(p) * 0.01)
        for n, p in net.named_parameters():
            if n.endswith("bias"):
                p.add_(torch.randn_like(p) * 0.05)
    net.deformation_net.set_aabb([1.4, 1.3, 1.45], [-1.35, -1.4, -1.2])
    return net


def _inputs(P, seed=1):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(P, 3, generator=g) * 3.4 - 1.7).cuda()
    scales = (torch.randn(P, 3, generator=g) * 0.6 - 5).cuda()
    rot = torch.randn(P, 4, generator=g).cuda()
    opacity = torch.randn(P, 1, generator=g).cuda()
    shs = torch.randn(P, 16, 3, generator=g).cuda()
    flow = (torch.randn(P, 3, generator=g) * 1e-3).cuda()
    return xyz, scales, rot, opacity, shs, flow


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


FIELD_CASES = [(5000, False, "op+sh"), (-5000, False, "op+sh"), (5000, False, "op"), (5000, False, "sh"),
               (40003, False, "op+sh"), (-40003, False, "op+sh"), (1000000, False, "op+sh"), (-1000000, False, "op+sh")]


@pytest.mark.gpu
@pytest.mark.parametrize("P,_unused,heads", FIELD_CASES, ids=[f"{P}-{h}" for P, _, h in FIELD_CASES])
def test_field_with_heads_matches_restatement(P, _unused, heads):
    """Every output and gradient against the restatement above (FP32 at small sizes, the FP64-anchored bar at 1M points); P < 0: one
    timestamp per point, else the camera's one timestamp (the shared spatial product under autograd)."""
    per_point = P < 0
    P = abs(P)
    no_do, no_dshs = not HEAD_MASKS[heads][0], not HEAD_MASKS[heads][1]
    net = _model(no_do, no_dshs)
    xyz, scales, rot, opacity, shs, flow = _inputs(P)
    time = torch.rand(P, 1, generator=torch.Generator().manual_seed(9)).cuda() if per_point else torch.full((P, 1), 0.37, device="cuda")
    fn = torch.tensor(22, device="cuda")
    sd = {k: v.detach().clone().contiguous().requires_grad_(v.dtype.is_floating_point) for k, v in net.state_dict().items()}
    a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot, opacity, shs)]
    out = net(a[0], a[1], a[2], a[3], a[4], time, flow, fn, 1)
    b = [t.clone().requires_grad_(True) for t in (xyz, scales, rot, opacity, shs)]
    ref = deform_forward(sd, 2, b[0], b[1], b[2], b[3], b[4], time, flow, fn, 1, no_do=no_do, no_dshs=no_dshs)
    for o, q in zip(out, ref):
        assert _rel(o, q) < 2e-5
    if no_do:
        assert torch.equal(out[3], opacity)
    if no_dshs:
        assert out[4] is a[4]
    g = torch.Generator().manual_seed(5)
    ws = [torch.randn(t.shape, generator=g).cuda() for t in out]
    sum(((o * w).sum() for o, w in zip(out, ws))).backward()
    sum(((o * w).sum() for o, w in zip(ref, ws))).backward()
    big = P >= 100000
    if big:
        d = torch.float64
        sd64 = {k: (v.detach().clone().to(d) if v.dtype.is_floating_point else v.detach().clone()).contiguous().requires_grad_(v.dtype.is_floating_point)
                for k, v in net.state_dict().items()}
        c = [t.clone().to(d).requires_grad_(True) for t in (xyz, scales, rot, opacity, shs)]
        q64 = deform_forward(sd64, 2, c[0], c[1], c[2], c[3], c[4], time.to(d), flow.to(d), fn, 1, no_do=no_do, no_dshs=no_dshs)
        sum(((o * w.to(d)).sum() for o, w in zip(q64, ws))).backward()
    for i, name in enumerate(("xyz", "scales", "rot", "opacity", "shs")):
        if not big:
            assert _rel(a[i].grad, b[i].grad) < 1e-3, name
        else:
            err = (a[i].grad - b[i].grad).reshape(P, -1).abs().max(dim=1).values / b[i].grad.abs().max()
            bad = err > 1e-3
            assert bad.float().mean().item() < 2e-4, (name, int(bad.sum()))
    params = dict(net.named_parameters())
    checked = 0
    for k, v in sd.items():
        if not v.requires_grad or k.endswith("grid.aabb") or k not in params:
            continue
        p = params[k]
        if v.grad is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            continue
        assert p.grad is not None, k
        if not big:
            assert _rel(p.grad, v.grad) < 1e-3, (k, _rel(p.grad, v.grad))
        else:
            ref64 = sd64[k].grad
            scale = ref64.abs().max()
            e_ours = ((p.grad.double() - ref64).abs().max() / scale).item()
            e_t32 = ((v.grad.double() - ref64).abs().max() / scale).item()
            assert e_ours <= max(1e-3, 2.0 * e_t32), (k, e_ours, e_t32)
        checked += 1
    n_heads = 3 + (not no_do) + (not no_dshs)
    assert checked >= 2 + 4 * n_heads + 12
    assert all(p.grad is None for n, p in net.named_parameters()
               if n.startswith("timenet") or (no_do and "opacity_deform" in n) or (no_dshs and "shs_deform" in n))


@pytest.mark.gpu
def test_field_heads_inference_and_counters():
    """No-grad forward bit-identical to the training forward (with and without a shared spatial product, which only
    re-associates the HexPlane product); the heads kernels run exactly when a head is on."""
    from b200gs import field
    P = 20011
    xyz, scales, rot, opacity, shs, flow = _inputs(P)
    fn = torch.tensor(7, device="cuda")
    net = _model(False, False)
    keep = field.AUTOGRAD_SPATIAL_SHARING
    field.AUTOGRAD_SPATIAL_SHARING = False
    try:
        a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot, opacity, shs)]
        train = net(*a, 0.61, flow, fn, 1)
    finally:
        field.AUTOGRAD_SPATIAL_SHARING = keep
    with torch.no_grad():
        infer = net(xyz, scales, rot, opacity, shs, 0.61, flow, fn, 1)
        with field.shared_spatial_product(net, xyz):
            shared = net(xyz, scales, rot, opacity, shs, 0.61, flow, fn, 1)
    for t, i, s in zip(train, infer, shared):
        assert torch.equal(t.detach(), i)
        assert _rel(s, i) < 2e-6
    # the heads' parameters must receive a gradient, the forward stash must have been kept for it
    sum(o.sum() for o in train).backward()
    assert all(p.grad is not None for n, p in net.named_parameters() if "opacity_deform" in n or "shs_deform" in n)
    off = _model(True, True)
    _lib.COUNTERS.clear()
    a = [t.clone().requires_grad_(True) for t in (xyz, scales, rot)]
    out = off(a[0], a[1], a[2], opacity, shs, 0.61, flow, fn, 1)
    sum(o.sum() for o in out[:3]).backward()
    assert _lib.COUNTERS["deform_heads_forward"] == 0 and _lib.COUNTERS["deform_heads_backward"] == 0
    out = net(a[0], a[1], a[2], opacity, shs, 0.61, flow, fn, 1)
    sum(o.sum() for o in out[:3]).backward()
    assert _lib.COUNTERS["deform_heads_forward"] == 1 and _lib.COUNTERS["deform_heads_backward"] == 1


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: trainer and rendering
def _gaussians(P, no_do, no_dshs, seed=3):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    raw = syn.make_gaussians(P, scale_mu=0.012, seed=seed, device="cpu")
    torch.manual_seed(0)
    h = engine.default_hyper()
    h.no_do, h.no_dshs = no_do, no_dshs
    m = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}, hyper=h).to(dev)
    with torch.no_grad():
        for p in m._deformation.deformation_net.grid.grids.parameters():
            p.add_(torch.randn_like(p) * 0.01)
        for n, p in m._deformation.named_parameters():
            if "opacity_deform" in n or "shs_deform" in n:
                p.mul_(3.0)                   # heads with a visible effect on the image
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("views", [1, 4])
def test_trainer_fast_path_with_heads_equals_plain_autograd(views):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    P, W, H = 30000, 240, 144
    ma = _gaussians(P, False, False)
    mb = copy.deepcopy(ma)
    ma.training_setup(); mb.training_setup()
    bg = torch.tensor([0.05, 0.1, 0.15], device=dev)
    h = engine.default_hyper()
    reg = (h.time_smoothness_weight, h.l1_time_planes, h.plane_tv_weight)
    ta = engine.ViewParallelTrainer(ma, bg, stage="fine", regulation=reg)
    tb = engine.ViewParallelTrainer(mb, bg, stage="fine", regulation=reg, shared_shs=False,
                                    render_fn=lambda cam, m, b, st: engine.render(cam, m, b, stage=st))
    assert ta.pipeline_views and len(ta.sh_params) == 2
    heads_params = {n for n, _ in ma.named_parameters() if "opacity_deform" in n or "shs_deform" in n}
    assert len(heads_params) == 8 and all(any(p is q for q in ta.arena_params) for n, p in ma.named_parameters() if n in heads_params)
    cams = syn.orbit_cameras(views, W, H, device=dev)
    g = torch.Generator().manual_seed(1)
    gts = [torch.rand(3, H, W, generator=g).to(dev) for _ in cams]
    _lib.COUNTERS.clear()
    la = float(ta.step(cams, gts)); lb = float(tb.step(cams, gts))
    assert _lib.COUNTERS["deform_heads_backward"] == 2 * views
    assert abs(la - lb) <= 2e-6 * max(1.0, abs(lb)), (la, lb)
    na = dict(ma.named_parameters())
    for n, q in mb.named_parameters():
        p = na[n]
        if q.grad is None:
            assert p.grad is None or n in ("_features_dc", "_features_rest"), n
            continue
        gp = ta.sh_grad[:, :1] if n == "_features_dc" else ta.sh_grad[:, 1:] if n == "_features_rest" else p.grad
        assert gp is not None, n
        if float(q.grad.abs().max()) == 0.0:
            assert float(gp.abs().max()) == 0.0, n
        else:
            assert _rel(gp, q.grad) <= 2e-5, (n, _rel(gp, q.grad))
    assert float(ta.sh_grad.abs().max()) > 0
    assert _rel(ta.viewspace_grad, tb.viewspace_grad) <= 2e-5
    for (n, p), (_, q) in zip(ma.named_parameters(), mb.named_parameters()):
        d = (p.detach() - q.detach()).abs()
        assert (d > 1e-6).float().mean().item() < 2e-3, (n, d.max().item())


@pytest.mark.gpu
def test_render_frames_with_heads_equals_frame_by_frame():
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    m = _gaussians(30000, False, False, seed=5)
    bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    cams = [syn.make_camera(200, 120, time=0.2 + 0.3 * i, frame_num=i, device=dev) for i in range(3)]
    with torch.no_grad():
        single = [engine.render(c, m, bg)["render"].clone() for c in cams]
    _lib.COUNTERS.clear()
    seq = [o for o in engine.render_frames(cams, m, bg)]
    # the shared spatial product re-associates the HexPlane product in FP32 (tests/test_render_sequence_parity.py), which can
    # flip an alpha < 1/255 for a handful of splats: the criterion of that test and of smoke()
    for a, b in zip(seq, single):
        diff = (a["render"] - b).abs().amax(dim=0)
        assert float((diff > 1e-4).float().mean()) < 1e-4, float(diff.max())
    assert _lib.COUNTERS["deform_heads_forward"] == len(cams) and _lib.COUNTERS["spatial_product_evaluations"] == 1
