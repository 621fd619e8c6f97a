"""GPU: engine.render_frames (spatial HexPlane product evaluated once for a sequence of frames, time planes per frame)
against engine.render frame by frame (the six-plane pass of the reference's render loop, render_4DGS.py:41-76).  The two differ
by FP32 re-association inside the field (<= 2e-6 on the features, tests/test_hexplane_split_parity.py), which can flip an
alpha < 1/255 or a tile-overlap decision for a handful of splats, so the image criterion is the one smoke() uses: all but
1e-4 of the pixels within 1e-4, and essentially all radii equal.
First passed on a B200 in round 2 (gpurun_out/pytest_r2a.log); part of the default `pytest -m gpu` since."""

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("streams", [1, 2, 3])
def test_render_frames_matches_frame_by_frame_rendering(streams):
    from b200gs import engine, synthetic as syn
    dev = torch.device("cuda", 0)
    P, W, H = 50000, 320, 200
    raw = syn.make_gaussians(P, scale_mu=0.01, seed=21, device="cpu")
    torch.manual_seed(0)
    model = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}).to(dev)
    with torch.no_grad():
        for p in model._deformation.deformation_net.grid.grids.parameters():
            p.add_(torch.randn_like(p) * 0.01)            # non-trivial time planes (SURVEY 8d)
    bg = torch.tensor([0.1, 0.2, 0.3], device=dev)
    cams = syn.orbit_cameras(7, W, H, device=dev)
    with torch.no_grad():
        ref = [engine.render(c, model, bg, stage="fine") for c in cams]
    # frames alternate over `streams` side streams; the consumer (here: a copy on the caller's stream) needs no stream handling
    seq = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in f.items()}
           for f in engine.render_frames(cams, model, bg, stage="fine", streams=streams)]
    from b200gs import field
    assert field._SHARED is None                           # the block cleaned up after itself
    one = list(engine.render_frames(cams, model, bg, stage="fine", streams=1))
    for a, b in zip(one, seq):                             # the stream layout changes nothing: bit-identical frames
        assert torch.equal(a["render"], b["render"]) and torch.equal(a["radii"], b["radii"]) and torch.equal(a["depth"], b["depth"])
    for a, b in zip(ref, seq):
        diff = (a["render"] - b["render"]).abs().amax(dim=0)
        assert float((diff > 1e-4).float().mean()) < 1e-4, float(diff.max())
        assert float((a["radii"] != b["radii"]).float().mean()) < 1e-4
        ddiff = (a["depth"] - b["depth"]).abs()
        assert float((ddiff > 1e-3).float().mean()) < 1e-4, float(ddiff.max())


def test_render_frames_matches_the_reference_stack(request):
    """The sequence path against the ORACLE stack (the reference's own CUDA rasterizer + the PyTorch field restatement pinned
    to the real scene/deformation.py, bench.make_reference_trainer), frame by frame: colour within 1e-4 on all but 1e-4 of the
    pixels (the fields agree to FP32 summation order, which can move a radius across an integer for a handful of splats).
    The oracle stack's frames are stored in tests/golden/parity_test_render_sequence_parity.npz (see tests/ref_golden.py), so
    the fractions are taken over the stored sample of each frame."""
    import types
    import bench
    from b200gs import engine
    from ref_golden import Golden
    ref = Golden(request)
    dev = torch.device("cuda", 0)
    args = types.SimpleNamespace(points=40000, width=320, height=192, views_per_gpu=5, scale_mu=0.01)
    raw, cams, _, _ = bench.build_scene(args, dev, 1, 0, "b200")
    ours_model, ours = bench.make_b200_trainer(args, raw, dev, 1, 0)
    seq = list(engine.render_frames(cams, ours_model, ours.bg, stage="fine"))
    for i, got in enumerate(seq):
        a, b = ref.sampled(f"frame{i}.render", got["render"])
        diff = np.abs(a - b)
        assert float((diff > 1e-4).mean()) < 1e-4, float(diff.max())
        a, b = ref.sampled(f"frame{i}.radii", got["radii"])
        assert float((a != b).mean()) < 1e-4
        a, b = ref.sampled(f"frame{i}.depth", got["depth"])
        ddiff = np.abs(a - b)
        assert float((ddiff > 1e-3).mean()) < 1e-4, float(ddiff.max())


def test_implicit_inference_cache_matches_and_is_dropped_by_fused_adam():
    """field.INFERENCE_SPATIAL_CACHE: the same reuse without a wrapper around the frame loop (unchanged render_4DGS.py through the
    launcher); a FusedAdam step must drop the cached product, a changed plane must miss it."""
    from b200gs import engine, field, synthetic as syn
    dev = torch.device("cuda", 0)
    P, W, H = 30000, 256, 160
    raw = syn.make_gaussians(P, scale_mu=0.01, seed=22, device="cpu")
    torch.manual_seed(0)
    model = engine.GaussianState({k: v.to(dev) for k, v in raw.items()}).to(dev)
    model.training_setup()
    bg = torch.zeros(3, device=dev)
    cams = syn.orbit_cameras(3, W, H, device=dev)
    with torch.no_grad():
        ref = [engine.render(c, model, bg, stage="fine")["render"].clone() for c in cams]
    field.INFERENCE_SPATIAL_CACHE = True
    try:
        with torch.no_grad():
            got = [engine.render(c, model, bg, stage="fine")["render"].clone() for c in cams]
        assert field._INFER is not None
        for a, b in zip(ref, got):
            assert float(((a - b).abs().amax(dim=0) > 1e-4).float().mean()) < 1e-4
        tr = engine.ViewParallelTrainer(model, bg)
        tr.step(cams[:2], [torch.rand(3, H, W, device=dev) for _ in range(2)])
        assert field._INFER is None                           # FusedAdam.step dropped it
        with torch.no_grad():
            after = engine.render(cams[0], model, bg, stage="fine")["render"]
            key = field._INFER.key
            next(iter(model._deformation.deformation_net.grid.grids.parameters())).add_(0.01)      # version bump
            engine.render(cams[0], model, bg, stage="fine")
            assert field._INFER.key != key
        assert float((after - ref[0]).abs().max()) > 0        # the parameters did move
    finally:
        field.INFERENCE_SPATIAL_CACHE = False
        field.invalidate_inference_cache()
