"""The deformation-MLP kernels (b200gs_deform_mlp_forward / _backward, include/b200gs.h) called directly through ctypes and
compared element by element with an FP64 restatement of csrc/deform_mlp.cu:5-10 and its derivative.

Metric: |y - y64| <= eps * M for every element, where M is the same FP64 chain evaluated on |W|, |b| and |activations| with
the FP64 ReLU masks applied (for the outputs plus |xyz|, |scales|, |rot| and |delta * frame_num * flow|).  The inputs are
drawn with a ReLU margin (every hidden and head pre-activation at least 1e-4 of its layer's scale away from 0), so the ReLU
masks of FP64 and of the kernels agree and every element can be held to the bound at every point count.

  forward outputs, d_features     eps = 2^-17   the three-term TF32 split (lo*hi + hi*lo + hi*hi) reproduces FP32 products to
                                                ~2^-21 relative; the rest is FP32 accumulation.  A single-pass TF32 product
                                                (2^-11) is ~2^6 over the bound.
  weight / bias gradients, FP64   eps = 2^-9    X is rounded to TF32 once (2^-11 per term).
  weight / bias gradients,        eps = 2^-16   against the MODELLED reference of what the kernels round (P >= 1024): dY
    modelled                                    exact, X rounded to TF32 with cvt.rna.  Both backwards keep dY as an exact
                                                hi + lo pair.  dW1 = dh^T tf32(feature) and dW2 = dz^T tf32(relu(hidden)) in both;
                                                dW3 = d_out^T relu(z) is plain FP32 in the tcgen05 backward (feature dim 64) and
                                                d_out^T tf32(relu(z)) in the mma.sync backward (feature dim 128); bias gradients
                                                are plain FP32 sums in both.  X is the value the forward stashed, so the model
                                                rounds exactly what the kernel rounded.
"""
import ctypes
import math

import pytest
import torch

from b200gs import _lib
from b200gs.field import _MlpGrads, _MlpWeights

MW = 64
KD = (3, 3, 4)
EPS_FWD = 2.0 ** -17
EPS_W64 = 2.0 ** -9
EPS_WMOD = 2.0 ** -16
MODELLED_MIN_P = 1024           # below this a weight-gradient sum has too few terms for the modelled tier to mean more than FP64's
FN, DELTA = 22.0, 0.37
SENTINEL = -12345.5             # written past the end of every output buffer; must survive
DEAD_H = (3, 40)                # hidden units with zero W1 row and b1 entry: exactly 0 for every point
DEAD_Z = (11, 18, 25)           # head h: unit DEAD_Z[h] of its hidden layer has a zero W2 row and b2 entry
NAMES = ("w1", "b1") + tuple(f"{n}_{h}" for h in range(3) for n in ("w2", "b2", "w3", "b3"))


# ---------------------------------------------------------------------------------------------------------------------------
# reference
def tf32_rna(x):
    """cvt.rna.tf32.f32: round an FP32 tensor to 10 explicit mantissa bits, ties away from zero."""
    b = x.contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def tf32_trunc(x):
    """What a tensor core reads from an FP32 container: the low 13 mantissa bits dropped."""
    return (x.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def stash_index(P, cols=MW):
    """Index of element (row, col) in one plane of the activation stash / the tiled feature layout (tc5_common.cuh stash_off)."""
    r = torch.arange(P, dtype=torch.int64)[:, None]
    c = torch.arange(cols, dtype=torch.int64)[None, :]
    return (r >> 7) * (128 * MW) + ((r & 127) >> 2) * 256 + (c >> 2) * 16 + (r & 3) * 4 + (c & 3)


def stash_plane_floats(P):
    return (P + 127) // 128 * 128 * MW


def make_weights(F, seed):
    """nn.Linear-style weights of all three heads with non-trivial biases and the dead units above (float32, CPU)."""
    g = torch.Generator().manual_seed(seed)

    def lin(o, i):
        bd = 1.0 / math.sqrt(i)
        return ((torch.rand(o, i, generator=g) * 2 - 1) * bd,
                (torch.rand(o, generator=g) * 2 - 1) * bd + torch.randn(o, generator=g) * 0.05)
    W = {}
    W["w1"], W["b1"] = lin(MW, F)
    W["w1"][list(DEAD_H)] = 0.0
    W["b1"][list(DEAD_H)] = 0.0
    for h in range(3):
        w2, b2 = lin(MW, MW)
        w2[DEAD_Z[h]] = 0.0
        b2[DEAD_Z[h]] = 0.0
        W[f"w2_{h}"], W[f"b2_{h}"] = w2, b2
        W[f"w3_{h}"], W[f"b3_{h}"] = lin(KD[h], MW)
    return W


def mlp(W, x, heads, dtype=torch.float64, rnd=None, magnitudes=False):
    """Forward and backward of the deformation MLP in `dtype` (every input is cast first).  rnd: optional rounding applied to
    both operands of every product (emulates a reduced-precision kernel).  magnitudes: also return M of every quantity, the
    same chain on |W|, |b| and |activations| under the ReLU masks of this evaluation."""
    W = {k: v.to(device=x["feat"].device, dtype=dtype) for k, v in W.items()}
    x = {k: [t.to(dtype) for t in v] if isinstance(v, list) else v.to(dtype) if torch.is_tensor(v) else v for k, v in x.items()}
    rnd = rnd or (lambda t: t)
    mm = lambda a, b: rnd(a) @ rnd(b)
    out, M = {}, {}
    feat = x["feat"]
    a1 = mm(feat, W["w1"].T) + W["b1"]
    m1 = (a1 > 0).to(dtype)
    out["h"] = a1 * m1
    if magnitudes:
        Mh = (feat.abs() @ W["w1"].abs().T + W["b1"].abs()) * m1
    d_rh = torch.zeros_like(a1)
    Md_rh = torch.zeros_like(a1)
    pass_in = (x["xyz"], x["scales"], x["rot"])
    for h in range(3):
        name = ("pts", "scales", "rot")[h]
        if not heads[h]:
            out[name] = pass_in[h].clone()
            M[name] = pass_in[h].abs()
            continue
        w2, b2, w3, b3 = (W[f"{n}_{h}"] for n in ("w2", "b2", "w3", "b3"))
        a2 = mm(out["h"], w2.T) + b2
        m2 = (a2 > 0).to(dtype)
        z = a2 * m2
        out[f"z_{h}"] = z
        o = mm(z, w3.T) + b3
        dout = x["dout"][h]
        dz = mm(dout, w3) * m2
        d_rh = d_rh + mm(dz, w2)
        out[f"w3_{h}"] = dout.T @ z
        out[f"b3_{h}"] = dout.sum(0)
        out[f"w2_{h}"] = dz.T @ out["h"]
        out[f"b2_{h}"] = dz.sum(0)
        if magnitudes:
            Mz = (Mh @ w2.abs().T + b2.abs()) * m2
            Mo = Mz @ w3.abs().T + b3.abs()
            Mdz = (dout.abs() @ w3.abs()) * m2
            Md_rh = Md_rh + Mdz @ w2.abs()
            M[f"w3_{h}"] = dout.abs().T @ Mz
            M[f"b3_{h}"] = dout.abs().sum(0)
            M[f"w2_{h}"] = Mdz.T @ Mh
            M[f"b2_{h}"] = Mdz.sum(0)
            M[f"dz_{h}"] = Mdz
        out[f"dz_{h}"] = dz
        if h == 0:
            flow = x["delta"] * (x["fn"] * x["flow"])
            out[name] = x["xyz"] + (o + flow)
            if magnitudes:
                M[name] = x["xyz"].abs() + Mo + flow.abs()
        else:
            out[name] = pass_in[h] + o
            if magnitudes:
                M[name] = pass_in[h].abs() + Mo
    dh = d_rh * m1
    out["dh"] = dh
    out["dfeat"] = mm(dh, W["w1"])
    out["w1"] = dh.T @ feat
    out["b1"] = dh.sum(0)
    if magnitudes:
        Mdh = Md_rh * m1
        M["dfeat"] = Mdh @ W["w1"].abs()
        M["w1"] = Mdh.T @ feat.abs()
        M["b1"] = Mdh.sum(0)
        M["dh"] = Mdh
    return out, M


def modelled_grads(ref, x, heads, stash_h, stash_z, tf32_w3):
    """The weight gradients the backward kernels compute, in FP64: dY exact (FP64), X = the stashed FP32 activation or the
    feature, rounded to TF32 (cvt.rna) where the kernel rounds it.  Bias gradients are exact sums."""
    d = torch.float64
    g = {"w1": ref["dh"].T @ tf32_rna(x["feat"]).to(d), "b1": ref["b1"]}
    for h in range(3):
        if not heads[h]:
            continue
        zx = tf32_rna(stash_z[h]) if tf32_w3 else stash_z[h]
        g[f"w3_{h}"] = x["dout"][h].to(d).T @ zx.to(d)
        g[f"b3_{h}"] = ref[f"b3_{h}"]
        g[f"w2_{h}"] = ref[f"dz_{h}"].T @ tf32_rna(stash_h).to(d)
        g[f"b2_{h}"] = ref[f"b2_{h}"]
    return g


def ratio(y, ref, M, eps):
    """max over elements of |y - ref| / (eps * M); an element with M == 0 must match exactly; NaN / inf count as infinite."""
    d = (y.to(torch.float64) - ref.to(torch.float64)).abs()
    lim = eps * M.to(torch.float64)
    r = torch.where(lim > 0, d / torch.where(lim > 0, lim, 1.0), torch.where(d > 0, math.inf, 0.0))
    r = torch.where(torch.isfinite(d), r, math.inf)
    return r.max().item() if r.numel() else 0.0


def draw_inputs(F, P, W, seed, device="cpu"):
    """P points whose hidden and head pre-activations all keep a ReLU margin (see the module docstring), plus the
    pass-through inputs and upstream gradients (biased towards positive, so weight-gradient sums do not cancel)."""
    g = torch.Generator().manual_seed(seed)
    Wd = {k: v.to(torch.float64) for k, v in W.items()}
    live_h = torch.ones(MW, dtype=torch.bool)
    live_h[list(DEAD_H)] = False
    kept = []
    n_kept = 0
    while n_kept < P:
        n = int(1.2 * (P - n_kept)) + 16
        feat = torch.randn(n, F, generator=g) * 0.6 + 0.15
        fd = feat.to(torch.float64)
        a1 = fd @ Wd["w1"].T + Wd["b1"]
        A1 = fd.abs() @ Wd["w1"].abs().T + Wd["b1"].abs()
        ok = ((a1.abs() >= 1e-4 * A1[:, live_h].mean()) | ~live_h).all(1)
        hdn = a1.clamp_min(0)
        Mh = A1 * (a1 > 0)
        for h in range(3):
            live_z = torch.ones(MW, dtype=torch.bool)
            live_z[DEAD_Z[h]] = False
            a2 = hdn @ Wd[f"w2_{h}"].T + Wd[f"b2_{h}"]
            A2 = Mh @ Wd[f"w2_{h}"].abs().T + Wd[f"b2_{h}"].abs()
            ok &= ((a2.abs() >= 1e-4 * A2[:, live_z].mean()) | ~live_z).all(1)
        kept.append(feat[ok])
        n_kept += int(ok.sum())
    x = {"feat": torch.cat(kept)[:P].contiguous(),
         "xyz": torch.rand(P, 3, generator=g) * 3.4 - 1.7,
         "scales": torch.randn(P, 3, generator=g) * 0.6 - 5,
         "rot": torch.randn(P, 4, generator=g),
         "flow": torch.randn(P, 3, generator=g) * 0.05,
         "dout": [torch.randn(P, k, generator=g) + 0.5 for k in KD],
         "fn": FN, "delta": DELTA}
    return {k: ([t.to(device) for t in v] if isinstance(v, list) else v.to(device) if torch.is_tensor(v) else v)
            for k, v in x.items()}


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: the metric tells a correct kernel from a subtly wrong one
def _cpu_case(P=2048, F=64):
    W = make_weights(F, 7)
    x = draw_inputs(F, P, W, 8)
    heads = (True, True, True)
    ref, M = mlp(W, x, heads, magnitudes=True)
    return W, x, heads, ref, M


def test_metric_accepts_fp32_and_rejects_single_pass_tf32_forward():
    W, x, heads, ref, M = _cpu_case()
    fp32, _ = mlp(W, x, heads, dtype=torch.float32)
    tf32, _ = mlp(W, x, heads, dtype=torch.float32, rnd=tf32_rna)
    for q in ("pts", "scales", "rot", "dfeat"):
        good, bad = ratio(fp32[q], ref[q], M[q], EPS_FWD), ratio(tf32[q], ref[q], M[q], EPS_FWD)
        print(f"{q}: fp32 {good:.3f}  1xTF32 {bad:.1f}")
        assert good < 0.05, (q, good)
        # the outputs' M includes the pass-through inputs (|scales| ~ 5 against head outputs ~ 0.3), which dilutes the head's
        # error; d_features has no such term
        assert bad > (4.0 if q == "dfeat" else 1.1), (q, bad)
    for q in [n for n in NAMES if n in ref]:
        assert ratio(fp32[q], ref[q], M[q], EPS_W64) < 0.05, q


def test_metric_rejects_weight_gradients_with_rounded_dy():
    """A backward that rounds dY to TF32 (drops the lo half of the split) instead of keeping it exact fails the modelled tier;
    the correct model passes it with margin."""
    W, x, heads, ref, M = _cpu_case()
    fp32, _ = mlp(W, x, heads, dtype=torch.float32)
    h32 = fp32["h"].to(torch.float32)
    mod = modelled_grads(ref, x, heads, h32, [fp32.get(f"z_{h}") for h in range(3)], tf32_w3=False)
    d = torch.float64
    for h in range(3):
        q = f"w2_{h}"
        dz32 = ref[f"dz_{h}"].to(torch.float32)
        exact = ref[f"dz_{h}"].T @ tf32_rna(h32).to(d)
        trunc = tf32_trunc(dz32).to(d).T @ tf32_rna(h32).to(d)
        rna = tf32_rna(dz32).to(d).T @ tf32_rna(h32).to(d)
        r_ok, r_trunc, r_rna = (ratio(v, mod[q], M[q], EPS_WMOD) for v in (exact, trunc, rna))
        print(f"{q}: exact dY {r_ok:.3f}  truncated dY {r_trunc:.1f}  rounded dY {r_rna:.2f}")
        assert r_ok < 0.05
        assert r_trunc > 2.0, (q, r_trunc)
        assert r_rna > 1.5, (q, r_rna)
        assert ratio(trunc, ref[q], M[q], EPS_W64) < 1.0      # ... which the FP64 tier alone cannot see


# ---------------------------------------------------------------------------------------------------------------------------
# CPU: argument validation (fake device pointers: nothing may be launched)
def _fake_weights(F=64, width=MW, tiled=0, heads=(True, True, True)):
    w = _MlpWeights(feat_dim=F, width=width, w1=0x10000, b1=0x20000, feat_tiled=tiled)
    for h in range(3):
        if heads[h]:
            w.w2[h], w.b2[h], w.w3[h], w.b3[h] = 0x30000 + 0x1000 * h, 0x40000 + 0x1000 * h, 0x50000 + 0x1000 * h, 0x60000 + 0x1000 * h
    return w


def _fake_grads():
    gw = _MlpGrads(w1=0x70000, b1=0x80000)
    for h in range(3):
        gw.w2[h], gw.b2[h], gw.w3[h], gw.b3[h] = 0x90000 + 0x1000 * h, 0xa0000 + 0x1000 * h, 0xb0000 + 0x1000 * h, 0xc0000 + 0x1000 * h
    return gw


def _fwd(L, w, P, saved=0xd0000):
    return L.b200gs_deform_mlp_forward(ctypes.byref(w), ctypes.c_longlong(P), 0xe0000, 0xe1000, 0xe2000, 0xe3000, 0xe4000, 1.0,
                                       None, 1.0, 0xe5000, 0xe6000, 0xe7000, saved, None)


def _bwd(L, w, P):
    return L.b200gs_deform_mlp_backward(ctypes.byref(w), ctypes.byref(_fake_grads()), ctypes.c_longlong(P), 0xe0000, 0xd0000,
                                        0xe1000, 0xe2000, 0xe3000, 0xe4000, None)


def test_mlp_entry_points_refuse_bad_arguments():
    L = _lib.lib()
    incomplete = _fake_weights()
    incomplete.b3[1] = None
    for what, w in (("net_width", _fake_weights(width=32)), ("feature dim", _fake_weights(F=96)),
                    ("tiled", _fake_weights(F=128, tiled=1)), ("head 1 incomplete", incomplete)):
        for call in (_fwd, _bwd):
            assert call(L, w, 1000) != 0, (what, call.__name__)
            assert what.encode() in L.b200gs_last_error(), (what, L.b200gs_last_error())
    # inference (nothing stashed) is the pipelined all-heads kernel only
    assert _fwd(L, _fake_weights(heads=(True, False, True)), 1000, saved=None) != 0
    assert b"needs all three heads" in L.b200gs_last_error()


def test_mlp_entry_points_return_early_for_empty_launches():
    """P <= 0 is a no-op: the fake pointers above would fault if anything touched them."""
    L = _lib.lib()
    for F, tiled in ((64, 0), (64, 1), (128, 0)):
        for P in (0, -1, -40003):
            assert _fwd(L, _fake_weights(F=F, tiled=tiled), P) == 0
            assert _fwd(L, _fake_weights(F=F, tiled=tiled, heads=(False, True, False)), P, saved=None) == 0
            assert _bwd(L, _fake_weights(F=F, tiled=tiled), P) == 0
    assert L.b200gs_deform_mlp_saved_floats(0) == 0 and L.b200gs_deform_mlp_saved_floats(-3) == 0
    assert L.b200gs_deform_mlp_saved_floats(129) == 4 * 256 * MW + 8 * MW * MW


# ---------------------------------------------------------------------------------------------------------------------------
# GPU: the kernels against the reference
LAYOUTS = ((64, False), (64, True), (128, False))
LAYOUT_IDS = ("F64", "F64tiled", "F128")
ALL_ON = (True, True, True)
NO_DS = (True, False, True)
MASKS = tuple(tuple(bool(m >> h & 1) for h in range(3)) for m in range(8))
EDGE_P = (1, 2, 3, 4, 5, 127, 128, 129, 255, 256, 257, 18944, 18945, 40003)     # 18944 = 148 tiles of 128: one per CTA
CASES = sorted({(m, P) for m in MASKS for P in (1, 129, 4099)} | {(m, P) for m in (ALL_ON, NO_DS) for P in EDGE_P},
               key=lambda c: (c[1], c[0]))


def _mask_id(heads):
    return "".join("xsr"[h] if heads[h] else "-" for h in range(3))


class Run:
    """One forward + backward through the C ABI with canaries around every buffer (see _launch)."""


def _launch(F, tiled, heads, P, W, x, *, fn_host=False, stash=True, backward=True, null_dout=(), null_off_grads=False,
            G0=None):
    """Inputs: NaN rows past P (tiled: NaN in the padding slots of the last tile and a whole NaN tile behind it).
    Outputs and stash: a SENTINEL tail that must survive.  d_features: NaN before the call (every row below P must come back
    finite), SENTINEL in every other slot.  Weight gradients: accumulated into G0 (their own 16-byte aligned buffers with a
    SENTINEL tail); the buffers of disabled heads are passed (holding G0) unless null_off_grads, and must stay untouched."""
    dev = torch.device("cuda")
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    nan = float("nan")
    r = Run()
    Wd = {k: v.to(dev).contiguous() for k, v in W.items()}

    def padded(t, fill=nan, extra=3):
        buf = torch.full((t.shape[0] + extra,) + tuple(t.shape[1:]), fill, dtype=torch.float32, device=dev)
        buf[:t.shape[0]] = t
        return buf

    n_tiles = (P + 127) // 128
    if tiled:
        idx = stash_index(P).to(dev)
        fbuf = torch.full(((n_tiles + 1) * 128 * MW,), nan, device=dev)
        fbuf[idx] = x["feat"].to(dev)
    else:
        fbuf = padded(x["feat"].to(dev))
    xyz, sc, rot, flow = (padded(x[k].to(dev)) for k in ("xyz", "scales", "rot", "flow"))
    outs = [torch.full((P + 2, k), SENTINEL, device=dev) for k in KD]
    n_saved = L.b200gs_deform_mlp_saved_floats(P)
    assert n_saved == 4 * stash_plane_floats(P) + 8 * MW * MW
    saved = None
    if stash:                       # NaN in the padding slots of the last stash tile, SENTINEL behind the buffer
        saved = torch.full((n_saved + 64,), nan, device=dev)
        saved[n_saved:] = SENTINEL
    fn_dev = torch.tensor([FN], device=dev)

    mw = _MlpWeights(feat_dim=F, width=MW, w1=Wd["w1"].data_ptr(), b1=Wd["b1"].data_ptr(), feat_tiled=int(tiled))
    for h in range(3):
        if heads[h]:
            mw.w2[h], mw.b2[h], mw.w3[h], mw.b3[h] = (Wd[f"{n}_{h}"].data_ptr() for n in ("w2", "b2", "w3", "b3"))
    rc = L.b200gs_deform_mlp_forward(ctypes.byref(mw), P, fbuf.data_ptr(), xyz.data_ptr(), sc.data_ptr(), rot.data_ptr(),
                                     flow.data_ptr(), FN if fn_host else 0.0, None if fn_host else fn_dev.data_ptr(), DELTA,
                                     outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(),
                                     saved.data_ptr() if saved is not None else None, stream)
    assert rc == 0, L.b200gs_last_error()
    torch.cuda.synchronize()
    for o in outs:
        assert bool((o[P:] == SENTINEL).all()), "forward wrote past row P"
    r.pts, r.scales, r.rot = (o[:P].clone() for o in outs)
    if saved is not None:
        assert bool((saved[n_saved:] == SENTINEL).all()), "forward wrote past b200gs_deform_mlp_saved_floats(P)"
        plane = stash_plane_floats(P)
        sidx = stash_index(P).to(dev)
        r.stash_h = saved[sidx].clone()
        r.stash_z = [saved[(1 + h) * plane + sidx].clone() if heads[h] else None for h in range(3)]
    if not backward:
        return r

    # backward
    if tiled:
        dfeat = torch.full(((n_tiles + 1) * 128 * MW,), SENTINEL, device=dev)
        dfeat[idx] = nan
    else:
        dfeat = torch.full((P + 3, F), SENTINEL, device=dev)
        dfeat[:P] = nan
    douts = [None if h in null_dout else padded(x["dout"][h].to(dev)) for h in range(3)]
    bufs = {}
    mg = _MlpGrads()
    for name in NAMES:
        h = int(name[-1]) if "_" in name else None
        shape = W[name].shape
        n = W[name].numel()
        buf = torch.full((n + 8,), SENTINEL, device=dev)
        buf[:n] = G0[name].to(dev).reshape(-1)
        bufs[name] = buf
        if h is not None and not heads[h] and null_off_grads:
            continue
        if h is None:
            setattr(mg, name, buf.data_ptr())
        else:
            getattr(mg, name.split("_")[0])[h] = buf.data_ptr()
    rc = L.b200gs_deform_mlp_backward(ctypes.byref(mw), ctypes.byref(mg), P, fbuf.data_ptr(), saved.data_ptr(),
                                      *[d.data_ptr() if d is not None else None for d in douts], dfeat.data_ptr(), stream)
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
    assert bool(torch.isfinite(r.dfeat).all()), "a d_features row below P was not written"
    r.gw = {}
    for name, buf in bufs.items():
        n = W[name].numel()
        assert bool((buf[n:] == SENTINEL).all()), f"backward wrote past the end of the {name} gradient"
        h = int(name[-1]) if "_" in name else None
        if h is not None and not heads[h]:
            assert torch.equal(buf[:n].cpu(), G0[name].reshape(-1)), f"gradient of disabled head {h} ({name}) was touched"
            continue
        r.gw[name] = buf[:n].reshape(W[name].shape).cpu()
    return r


_REF = {}


def _case(F, P, heads):
    """Weights, inputs, FP64 reference and the G0 fill of one case (cached: the contract tests reuse the matrix's cases)."""
    key = (F, P, heads)
    if key not in _REF:
        if len(_REF) > 8:
            _REF.clear()
        W = make_weights(F, 100 + F)
        x = draw_inputs(F, P, W, 1000 * F + P, device="cuda")
        ref, M = mlp(W, x, heads, magnitudes=True)
        ref = {k: v.cpu() for k, v in ref.items()}
        M = {k: v.cpu() for k, v in M.items()}
        g = torch.Generator().manual_seed(P)
        # G0 at 1/16 of each element's magnitude: a write instead of an add is 16x over any bound, while the FP32 rounding of
        # the running sum stays at the scale of the gradient itself (dead / disabled elements get the tensor's mean scale)
        G0 = {}
        for name in NAMES:
            m = M.get(name)
            m = m.to(torch.float32) if m is not None else torch.ones(W[name].shape)
            base = torch.where(m > 0, m, m.mean().clamp_min(1e-3))
            G0[name] = (base * (torch.rand(W[name].shape, generator=g) + 0.5) / 16 *
                        torch.sign(torch.randn(W[name].shape, generator=g))).to(torch.float32)
        _REF[key] = (W, x, ref, M, G0)
    return _REF[key]


def _check(F, heads, P, r, ref, M, x, G0, label=""):
    """Every bound of the module docstring, plus the dead units' exact zeros; returns {quantity: worst ratio}."""
    worst = {}
    for q, y in (("pts", r.pts), ("scales", r.scales), ("rot", r.rot)):
        worst[q] = ratio(y.cpu(), ref[q], M[q], EPS_FWD)
        h = ("pts", "scales", "rot").index(q)
        if not heads[h]:
            assert torch.equal(y.cpu(), x[("xyz", "scales", "rot")[h]].cpu()), f"disabled head {h} must pass {q} through"
    worst["dfeat"] = ratio(r.dfeat.cpu(), ref["dfeat"], M["dfeat"], EPS_FWD)
    d64 = {k: v.to(torch.float64) - G0[k].to(torch.float64) for k, v in r.gw.items()}
    for k, v in d64.items():
        worst["fp64:" + k.split("_")[0]] = max(worst.get("fp64:" + k.split("_")[0], 0.0), ratio(v, ref[k], M[k], EPS_W64))
    if P >= MODELLED_MIN_P:
        xs = {"feat": x["feat"].cpu(), "dout": [t.cpu() for t in x["dout"]]}
        mod = modelled_grads(ref, xs, heads, r.stash_h.cpu(), [z.cpu() if z is not None else None for z in r.stash_z],
                             tf32_w3=(F == 128))
        for k, v in d64.items():
            worst["mod:" + k.split("_")[0]] = max(worst.get("mod:" + k.split("_")[0], 0.0), ratio(v, mod[k], M[k], EPS_WMOD))
    print(f"[deform-mlp F={F} heads={_mask_id(heads)} P={P}{label}] " + " ".join(f"{k}={v:.3g}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v <= 1.0}
    assert not bad, bad
    # dead units: exactly nothing is added
    dead_h = list(DEAD_H)
    exact = [("w1", (dead_h, slice(None))), ("b1", (dead_h,))]
    for h in range(3):
        if heads[h]:
            exact += [(f"w2_{h}", (slice(None), dead_h)), (f"w2_{h}", (DEAD_Z[h], slice(None))), (f"b2_{h}", (DEAD_Z[h],)),
                      (f"w3_{h}", (slice(None), DEAD_Z[h]))]
    for k, ix in exact:
        assert torch.equal(r.gw[k][ix], G0[k][ix]), f"{k}: a dead unit's gradient is not exactly 0"
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("F,tiled", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("heads,P", CASES, ids=[f"{_mask_id(m)}-P{P}" for m, P in CASES])
def test_deform_mlp_matches_fp64(F, tiled, heads, P):
    W, x, ref, M, G0 = _case(F, P, heads)
    r = _launch(F, tiled, heads, P, W, x, G0=G0, null_off_grads=(P % 2 == 0))
    _check(F, heads, P, r, ref, M, x, G0)


@pytest.mark.gpu
@pytest.mark.parametrize("F,tiled", LAYOUTS, ids=LAYOUT_IDS)
def test_deform_mlp_contract(F, tiled):
    """Null upstream gradients = zeros; frame_num by host value = by device pointer; inference (saved = NULL) = stashed;
    two calls give the same bits; forward outputs and d_features do not depend on the SM caps, weight gradients stay in the
    modelled tier under them."""
    P = 18945
    L = _lib.lib()
    W, x, ref, M, G0 = _case(F, P, ALL_ON)
    base = _launch(F, tiled, ALL_ON, P, W, x, G0=G0)
    _check(F, ALL_ON, P, base, ref, M, x, G0)
    again = _launch(F, tiled, ALL_ON, P, W, x, G0=G0)
    for q in ("pts", "scales", "rot", "dfeat"):
        assert torch.equal(getattr(again, q), getattr(base, q)), f"{q} differs between two identical calls"
    host = _launch(F, tiled, ALL_ON, P, W, x, fn_host=True, backward=False)
    infer = _launch(F, tiled, ALL_ON, P, W, x, stash=False, backward=False)
    for q in ("pts", "scales", "rot"):
        assert torch.equal(getattr(host, q), getattr(base, q)), f"{q}: frame_num by value differs from by pointer"
        assert torch.equal(getattr(infer, q), getattr(base, q)), f"{q}: inference forward differs from the stashing one"

    # null upstream gradients behave as zeros
    for nulls in ((0,), (1,), (2,), (0, 2)):
        xz = dict(x, dout=[torch.zeros_like(t) if h in nulls else t for h, t in enumerate(x["dout"])])
        refz, Mz = mlp(W, xz, ALL_ON, magnitudes=True)
        refz = {k: v.cpu() for k, v in refz.items()}
        Mz = {k: v.cpu() for k, v in Mz.items()}
        zeros = _launch(F, tiled, ALL_ON, P, W, xz, G0=G0)
        null = _launch(F, tiled, ALL_ON, P, W, x, G0=G0, null_dout=nulls)
        assert torch.equal(null.dfeat, zeros.dfeat), nulls
        _check(F, ALL_ON, P, null, refz, Mz, xz, G0, label=f" null d_out {nulls}")

    # SM caps (the forward honours mlp_fwd_sms; the tcgen05 backward mlp_bwd_sms, the feature-dim-128 backward ignores it)
    try:
        for cap in (1, 7, 120, 147):
            assert L.b200gs_set_option(b"mlp_fwd_sms", cap) == 0 and L.b200gs_set_option(b"mlp_bwd_sms", cap) == 0
            capped = _launch(F, tiled, ALL_ON, P, W, x, G0=G0)
            for q in ("pts", "scales", "rot", "dfeat"):
                assert torch.equal(getattr(capped, q), getattr(base, q)), f"{q} changes with {cap} CTAs"
            _check(F, ALL_ON, P, capped, ref, M, x, G0, label=f" sms={cap}")
    finally:
        L.b200gs_set_option(b"mlp_fwd_sms", 0)
        L.b200gs_set_option(b"mlp_bwd_sms", 0)
