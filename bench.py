#!/usr/bin/env python
"""Headline benchmark: 4DGS training throughput, 1M Gaussians, 1280x720, a batch of 8 views per optimiser step
(BASELINE.json C3: "8 views over N x B200").

    python bench.py --gpus N --steps K --warmup W              # this repo (sm_100a kernels via the C ABI)
    python bench.py --impl reference --gpus N --steps K ...    # the reference's own code path

One step = one fine-stage training iteration over the GLOBAL batch of 8 views (train_4DGS.py:172-297): per view HexPlane
deformation -> exp/normalize/sigmoid -> rasterize -> L1 -> backward through all of it; then the gradient exchange
(N > 1: NCCL all-reduce of the SH gradient on a side stream + of the flat arena), the plane regulariser and one fused Adam
step over every parameter.  The 8 views are sharded over the ranks (8 / 4 / 2 / 1 views per GPU): STRONG scaling, the
configuration BASELINE.json names.  `value` = view-iterations per second of the whole job, timed on the device with CUDA events
between barriers, max over ranks.  For N > 1 a second block (`weak`) repeats the measurement with 8 views PER GPU.
`e2e` repeats the measurement through the same public API with the ground-truth images in pinned HOST memory as the dataset
holds them (uint8 HWC), uploaded inside the timed region every step (prefetched on a side stream), and the loss read back to
the host every step (asynchronously, through a pinned ring).

Side blocks in the same JSON line: `render` (BASELINE config 4: five 60-frame camera paths at 1920x1080 and 1280x720, frames
sharded over ranks), `raster_only` (config 2: rasterizer fwd+bwd alone at 200k / 512^2 and 1M / 720p), `kernels` (live
per-kernel durations and roofline fractions), `timeline` (where a step's time goes, CUDA events), `cpu_baseline`
(config 1 + a CPU port of one view-iteration, timed on the host cores after the timed region).

The reference arm runs the reference's own CUDA rasterizer (oracle/_ref/libref_rast.so, built unmodified from
/root/reference by oracle/build_ref.sh), a plain-PyTorch port of its HexPlane / deformation modules (oracle/field_torch.py,
pinned bit-exact against the real modules) and torch.optim.Adam, on the same GPU, same scene, same loop.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written into it, bytecode caches included
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in ("iclr2025_3d-mom_b200", os.path.join("iclr2025_3d-mom_b200", "dropin"), "tests", ""):
    sys.path.insert(0, os.path.join(ROOT, p))

import torch  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cpu"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--width", type=int, default=1280)
    ap.add_argument("--height", type=int, default=720)
    ap.add_argument("--global-batch", type=int, default=8, help="views per optimiser step over ALL GPUs (BASELINE config 3: 8)")
    ap.add_argument("--views-per-gpu", type=int, default=8, help="per-GPU batch of the weak-scaling block (N > 1)")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling block at N > 1")
    ap.add_argument("--scale-mu", type=float, default=0.010, help="S-coarse 0.010 / S-fine 0.004 (SURVEY.md 8d)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--render-frames", type=int, default=60, help="frames per camera path of the render block (0 = skip)")
    ap.add_argument("--render-streams", type=int, default=2, help="streams engine.render_frames alternates the frames of a path over")
    ap.add_argument("--no-raster-only", action="store_true", help="skip the config-2 rasterizer-only block")
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 stress block (5M Gaussians at 3840x2160, N = 1 only)")
    ap.add_argument("--no-launcher-path", action="store_true", help="skip the block that runs the reference's unchanged train_4DGS.py through the launcher")
    ap.add_argument("--no-shared-spatial", action="store_true",
                    help="render every frame with the full six-plane HexPlane pass instead of sharing the spatial product over a sequence")
    ap.add_argument("--cpu-points", type=int, default=0, help="override the cpu_baseline sample size")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed to DIR/<name>.npy (see dump_outputs)")
    return ap.parse_args()


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, enabled=True):
        # rank 0 only at N > 1: eight processes forking nvidia-smi ten times a second contend for the driver and showed up as
        # straggling ranks (the timed value is the MAX over ranks); one sampler at 4 Hz sees the same clocks
        self.index, self.rows, self.stop, self.enabled = index, [], False, enabled
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.25)

    def __enter__(self):
        if self.enabled:
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.enabled:
            self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(self.rows), "reasons": sorted(reasons)}




def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "sm_max_mhz": 1965.0}, "fallback"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, keyed by kernel name, from the committed summary of the
    `ncu --set full` capture of THIS tree's default kernels (profiles/ncu_dram_bytes.json, written by tools/ncu_summary.py);
    {} when there is none -- `roofline.traffic` is then null rather than a stale constant."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_dram_bytes.json")))
        return {k: v for k, v in d.get("kernels", {}).items()}, d.get("source")
    except Exception:
        return {}, None


# ---------------------------------------------------------------------------------------------
def scene_images_u8(args, n_global):
    """Seeded ground-truth images the way the dataset holds them: uint8 [H,W,3] (PIL), one per view of the global batch."""
    g = torch.Generator().manual_seed(1234)
    return [(torch.rand(args.height, args.width, 3, generator=g) * 255.999).to(torch.uint8) for _ in range(n_global)]


def build_scene(args, device, world, rank, impl):
    """raw Gaussians, THIS rank's cameras, its ground-truth images as pinned float32 [3,H,W] host tensors
    (= u8 / 255 exactly as utils/general_utils.py:PILtoTorch converts them), and the global batch size."""
    from b200gs import synthetic as syn
    raw = syn.make_gaussians(args.points, scale_mu=args.scale_mu, device="cpu")
    n_global = getattr(args, "global_views", None) or args.views_per_gpu * world
    cams_all = syn.orbit_cameras(n_global, args.width, args.height, device=device)
    mine = list(range(rank, n_global, world))
    u8 = scene_images_u8(args, n_global)
    pin = (lambda t: t.pin_memory()) if torch.cuda.is_available() else (lambda t: t)
    gts_host = [pin((u8[b].float() / 255.0).permute(2, 0, 1).contiguous()) for b in mine]
    build_scene.last_u8 = [pin(u8[b].contiguous()) for b in mine]
    cams = [cams_all[b] for b in mine]
    return raw, cams, gts_host, n_global


def make_b200_trainer(args, raw, device, world, rank):
    from b200gs import engine
    torch.manual_seed(6666)
    model = engine.GaussianState({k: v.to(device) for k, v in raw.items()}, hyper=engine.default_hyper()).to(device)
    with torch.no_grad():
        xyz = model._xyz
        model._deformation.deformation_net.set_aabb(xyz.max(0).values.tolist(), xyz.min(0).values.tolist())   # scene/__init__.py:72-78
        for p in model._deformation.deformation_net.grid.grids.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    model.training_setup()
    pg = None
    bg = torch.zeros(3, device=device)
    h = engine.default_hyper()
    return model, engine.ViewParallelTrainer(model, bg, stage="fine", process_group=pg, world_size=world, rank=rank,
                                             regulation=(h.time_smoothness_weight, h.l1_time_planes, h.plane_tv_weight))


# ---- reference arm -------------------------------------------------------------------------------
def make_reference_trainer(args, raw, device, world, rank):
    """Reference code path on the GPU: unmodified reference CUDA rasterizer (oracle/_ref) behind a
    torch.autograd.Function that does what RAST/diff_gaussian_rasterization/__init__.py and
    rasterize_points.cu do (torch.zeros gradient tensors included), the PyTorch port of the
    HexPlane field, torch.optim.Adam, and the same loop as ViewParallelTrainer."""
    import ref_harness as rh
    from b200gs import engine
    from oracle import field_torch
    if not rh.have_ref():
        return None, None
    L = rh.rast()
    p = rh._p

    class RefRaster(torch.autograd.Function):
        @staticmethod
        def forward(ctx, means3D, means2D, sh, opac, scales, rots, cam, bg):
            P = means3D.shape[0]
            H, W = cam.image_height, cam.image_width
            color = torch.zeros(3, H, W, device=device); depth = torch.zeros(1, H, W, device=device)
            radii = torch.zeros(P, dtype=torch.int32, device=device)
            means3D, sh, opac, scales, rots = (t.contiguous() for t in (means3D, sh, opac, scales, rots))
            R = L.ref_rast_forward(P, 3, sh.shape[1], p(bg), W, H, p(means3D), p(sh), None, p(opac), p(scales), 1.0, p(rots), None,
                                   p(cam.viewmatrix), p(cam.projmatrix), p(cam.campos), cam.tanfovx, cam.tanfovy, 0, p(color),
                                   p(depth), p(radii), 0)
            assert R >= 0, L.ref_last_error()
            ctx.save_for_backward(means3D, sh, scales, rots, radii)
            ctx.cam, ctx.bg, ctx.R = cam, bg, R
            ctx.mark_non_differentiable(radii)
            return color, radii, depth

        @staticmethod
        def backward(ctx, dcolor, _dr, ddepth):
            means3D, sh, scales, rots, radii = ctx.saved_tensors
            cam, bg = ctx.cam, ctx.bg
            P = means3D.shape[0]; H, W = cam.image_height, cam.image_width
            z = lambda *s: torch.zeros(*s, device=device)
            g = dict(means2D=z(P, 3), conic=z(P, 2, 2), opacity=z(P, 1), colors=z(P, 3), depths=z(P, 1), means3D=z(P, 3),
                     cov3D=z(P, 6), sh=z(P, sh.shape[1], 3), scales=z(P, 3), rotations=z(P, 4))
            ddepth = ddepth.contiguous() if ddepth is not None else z(1, H, W)
            rc = L.ref_rast_backward(P, 3, sh.shape[1], ctx.R, p(bg), W, H, p(means3D), p(sh), None, p(scales), 1.0, p(rots), None,
                                     p(cam.viewmatrix), p(cam.projmatrix), p(cam.campos), cam.tanfovx, cam.tanfovy, p(radii),
                                     p(dcolor.contiguous()), p(ddepth), p(g["means2D"]), p(g["conic"]), p(g["opacity"]),
                                     p(g["colors"]), p(g["depths"]), p(g["means3D"]), p(g["cov3D"]), p(g["sh"]), p(g["scales"]),
                                     p(g["rotations"]), 0)
            assert rc == 0
            return g["means3D"], g["means2D"], g["sh"], g["opacity"], g["scales"], g["rotations"], None, None

    class RefModel(torch.nn.Module):
        def __init__(self):
            super().__init__()
            torch.manual_seed(6666)
            ours = engine.GaussianState({k: v for k, v in raw.items()}, hyper=engine.default_hyper())
            self._xyz, self._features_dc, self._features_rest = ours._xyz, ours._features_dc, ours._features_rest
            self._scaling, self._rotation, self._opacity = ours._scaling, ours._rotation, ours._opacity
            self.register_buffer("_scene_flow", ours._scene_flow)
            # same initial field parameters, held as plain contiguous tensors keyed like the state_dict
            self.field = torch.nn.ParameterDict()
            self.keys = {}
            for k, v in ours._deformation.state_dict().items():
                if v.dtype.is_floating_point and "poc" not in k:
                    name = k.replace(".", "__")
                    self.field[name] = torch.nn.Parameter(v.detach().clone().contiguous(), requires_grad=not k.endswith("aabb"))
                    self.keys[k] = name
            self.levels = len(ours._deformation.deformation_net.grid.grids)
            self.optimizer = None

        @property
        def get_xyz(self):
            return self._xyz

        def named_parameters(self, *a, **k):        # names as in the product model so the arena filter applies
            for n, q in super().named_parameters(*a, **k):
                yield ("_deformation." + n[len("field."):].replace("__", ".") if n.startswith("field.") else n), q

    model = RefModel().to(device)
    with torch.no_grad():
        xyz = model._xyz
        aabb = model.field[model.keys["deformation_net.grid.aabb"]]
        aabb.copy_(torch.stack([xyz.max(0).values, xyz.min(0).values]))
        torch.manual_seed(6666)
        for k, n in model.keys.items():
            if ".grids." in k:
                model.field[n].add_(torch.randn_like(model.field[n]) * 0.01)
    o = engine.default_opt()
    mlp = [q for k, n in model.keys.items() if "grid" not in k for q in [model.field[n]]]
    grid = [q for k, n in model.keys.items() if "grid" in k for q in [model.field[n]]]
    model.optimizer = torch.optim.Adam([
        {'params': [model._xyz], 'lr': o.position_lr_init, "name": "xyz"}, {'params': mlp, 'lr': o.deformation_lr_init, "name": "deformation"},
        {'params': grid, 'lr': o.grid_lr_init, "name": "grid"}, {'params': [model._features_dc], 'lr': o.feature_lr, "name": "f_dc"},
        {'params': [model._features_rest], 'lr': o.feature_lr / 20.0, "name": "f_rest"},
        {'params': [model._opacity], 'lr': o.opacity_lr, "name": "opacity"}, {'params': [model._scaling], 'lr': o.scaling_lr, "name": "scaling"},
        {'params': [model._rotation], 'lr': o.rotation_lr, "name": "rotation"}], lr=0.0, eps=1e-15)

    def ref_render(cam, m, bg, stage):
        P = m._xyz.shape[0]
        sp = torch.zeros_like(m._xyz, requires_grad=True)
        shs = torch.cat((m._features_dc, m._features_rest), dim=1)
        time_ = torch.full((P, 1), float(cam.time), device=device)
        sd = {k: m.field[n] for k, n in m.keys.items()}
        pts, sc, rt, op, sh = field_torch.deform_forward(sd, m.levels, m._xyz, m._scaling, m._rotation, m._opacity, shs, time_,
                                                         m._scene_flow, cam.frame_num, 1)
        color, radii, depth = RefRaster.apply(pts, sp, sh, torch.sigmoid(op), torch.exp(sc), torch.nn.functional.normalize(rt), cam, bg)
        return {"render": color, "viewspace_points": sp, "radii": radii, "depth": depth}

    def ref_regulation():
        """compute_regulation exactly as scene/gaussian_model.py:730-769 + scene/regulation.py:22-28 spell it (PyTorch ops)."""
        h = engine.default_hyper()
        grids = [[model.field[model.keys[f"deformation_net.grid.grids.{l}.{k}"]] for k in range(6)] for l in range(model.levels)]

        def smooth(t):
            hh = t.shape[2]
            first = t[..., 1:, :] - t[..., :hh - 1, :]
            second = first[..., 1:, :] - first[..., :hh - 2, :]
            return torch.square(second).mean()
        plane = sum(smooth(g[k]) for g in grids for k in (0, 1, 3))
        tsm = sum(smooth(g[k]) for g in grids for k in (2, 4, 5))
        l1 = sum(torch.abs(1 - g[k]).mean() for g in grids for k in (2, 4, 5))
        return h.plane_tv_weight * plane + h.time_smoothness_weight * tsm + h.l1_time_planes * l1

    bg = torch.zeros(3, device=device)
    return model, engine.ViewParallelTrainer(model, bg, stage="fine", world_size=world, rank=rank, render_fn=ref_render,
                                             regulation_fn=ref_regulation)


# ---- render FPS (BASELINE.json config 4) -------------------------------------------------------------
def render_block(args, model, device, world, rank, impl, ref_render=None):
    """Video rendering (render_4DGS.py:41-76): the five camera paths (up-down, side, zoom-in, circle, vfx; 60 frames each, time
    advancing along the path) of b200gs.synthetic.video_trajectories at 1920x1080 and 1280x720, frame f of path j on rank
    (60 j + f) mod N, no collective.  `fps` = frames per second on the device (deformation + rasterizer forward), `e2e_fps` adds
    the output path per frame: to8b + D2H into host memory (our arm: GPU quantise + async 3 B/pixel copy of every frame into its
    place in one pinned [frames,H,W,3] array, output.FrameStore -- `e2e_fps_ring_copy` is the older path through a 4-deep pinned
    ring with a host-side copy per frame; reference arm: the blocking float copy + host clip/cast of render_4DGS.py:49).  Pinned
    buffers are allocated once, before the timed loop."""
    import contextlib
    import numpy as np
    from b200gs import engine, synthetic as syn
    out = {}
    bg = torch.zeros(3, device=device)
    for tag, (W, H) in (("1920x1080", (1920, 1080)), ("1280x720", (args.width, args.height))):
        paths = syn.video_trajectories(W, H, frames=args.render_frames, device=device)
        # this rank's frames, grouped by path (a path is one sequence over the static model)
        mine, k = [], 0
        for name, cams in paths.items():
            sel = [c for i, c in enumerate(cams) if (k + i) % world == rank]
            k += len(cams)
            mine.append(sel)
        n_total = k
        fn = (lambda c: engine.render(c, model, bg, stage="fine")) if impl == "b200" else (lambda c: ref_render(c, model, bg, "fine"))

        def shared():
            if impl == "b200" and not args.no_shared_spatial:
                from b200gs import field as _field
                return _field.shared_spatial_product(model._deformation, model._xyz)
            return contextlib.nullcontext()

        def run_all(consume=None, streams=args.render_streams):
            for sel in mine:
                if impl == "b200" and not args.no_shared_spatial:
                    # the public sequence API: spatial half of the HexPlane field once per path, time planes per frame,
                    # consecutive frames alternating between two streams
                    for r in engine.render_frames(sel, model, bg, stage="fine", streams=streams):
                        if consume is not None:
                            consume(r["render"])
                    continue
                for c in sel:
                    r = fn(c)
                    if consume is not None:
                        consume(r["render"])
        with torch.no_grad():
            with shared():
                for c in mine[0][:3]:
                    fn(c)
            if impl == "b200" and not args.no_shared_spatial:      # warm both streams' allocator pools as well
                for _ in engine.render_frames(mine[0][:8], model, bg, stage="fine", streams=args.render_streams):
                    pass
            run_all()                                  # one untimed pass over every frame: the instance counts (binning buffers) grow
            torch.cuda.synchronize()                   # along a path, and the caching allocator should have seen the largest
            if world > 1:
                import torch.distributed as _dist
                _dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); run_all(); e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            ms_one_stream = None
            if impl == "b200" and not args.no_shared_spatial:          # the same without the two-stream frame pipelining
                e0.record(); run_all(streams=1); e1.record()
                torch.cuda.synchronize()
                ms_one_stream = e0.elapsed_time(e1)
            ms_plain = None
            if impl == "b200" and not args.no_shared_spatial:          # the same frames with the full six-plane pass per frame
                e0.record()
                for sel in mine:
                    for c in sel:
                        fn(c)
                e1.record()
                torch.cuda.synchronize()
                ms_plain = e0.elapsed_time(e1)
            frames_out = []
            if impl == "b200":
                from b200gs import output
                ring = output.FrameRing(H, W, depth=4, device=device)      # pinned buffers are allocated once, outside the loop
                ring.push(fn(mine[0][0])["render"]); ring.pop()

                def consume(img):
                    if ring.count == 4:
                        frames_out.append(ring.pop())
                    ring.push(img)
            else:
                def consume(img):
                    frames_out.append((255 * np.clip(img.cpu().numpy(), 0, 1)).astype(np.uint8))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run_all(consume)
            if impl == "b200":
                while ring.count:
                    frames_out.append(ring.pop())
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            del frames_out
            wall_ring = None
            if impl == "b200":
                del ring
                wall_ring = wall
                n_mine = sum(len(sel) for sel in mine)
                store = output.FrameStore(max(n_mine, 1), H, W, device=device)
                store.put(0, fn(mine[0][0])["render"]); store.array()
                slot = [0]

                def consume(img):
                    store.put(slot[0], img)
                    slot[0] += 1
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                run_all(consume)
                frames_arr = store.array()
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                assert frames_arr.shape[0] == max(n_mine, 1) and slot[0] == n_mine
                del frames_arr, store
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms, wall * 1e3, ms_plain if ms_plain is not None else 0.0,
                              wall_ring * 1e3 if wall_ring is not None else 0.0,
                              ms_one_stream if ms_one_stream is not None else 0.0], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
            if ms_plain is not None:
                ms_plain = float(t[2])
            if wall_ring is not None:
                wall_ring = float(t[3]) / 1e3
            if ms_one_stream is not None:
                ms_one_stream = float(t[4])
        out[tag] = {"fps": n_total / (ms / 1e3), "e2e_fps": n_total / wall, "frames": n_total, "paths": list(paths.keys()),
                    "d2h_bytes_per_frame": 3 * W * H if impl == "b200" else 12 * W * H}
        if ms_plain is not None:
            out[tag]["fps_full_field_per_frame"] = n_total / (ms_plain / 1e3)
        if ms_one_stream is not None:
            out[tag]["fps_one_stream"] = n_total / (ms_one_stream / 1e3)
        if wall_ring is not None:
            out[tag]["e2e_fps_ring_copy"] = n_total / wall_ring
    return out


# ---- rasterizer alone (BASELINE.json config 2) ---------------------------------------------------------
def raster_only_block(args, device, impl):
    """Static 3DGS rasterizer fwd+bwd through the rasterizer API alone (coarse-stage semantics: no deformation field), SH degree 3,
    at 200k Gaussians / 512x512 (config 2) and 1M / 1280x720, S-coarse scene, 5 warm-up + 20 timed repetitions, CUDA events.
    Our arm calls the drop-in's `_C` entry points; the reference arm its own CUDA code (oracle/_ref) with the torch.zeros fills
    its glue does (rasterize_points.cu:58-60, :154-163).  Same seeded inputs on both sides."""
    from b200gs import synthetic as syn
    out = {}
    E = torch.Tensor([])
    for tag, (P, W, H, mu) in (("200k_512x512", (200000, 512, 512, 0.010)), ("1M_1280x720", (1000000, 1280, 720, 0.010))):
        raw = syn.make_gaussians(P, scale_mu=mu, device=device); act = syn.activated(raw)
        cam = syn.make_camera(W, H, device=device)
        bg = torch.zeros(3, device=device)
        gt = torch.rand(3, H, W, device=device)
        dLd = torch.zeros(1, H, W, device=device)
        st = {}
        if impl == "b200":
            from b200gs.rasterizer import _C

            def fwd():
                st["o"] = _C.rasterize_gaussians(bg, act["means3D"], E, act["opacities"], act["scales"], act["rotations"], 1.0, E, cam.viewmatrix,
                                                 cam.projmatrix, cam.tanfovx, cam.tanfovy, H, W, act["shs"], 3, cam.campos, False, False)
            fwd()
            R, color, depth, radii, geom, binb, img = st["o"]
            dLc = torch.sign(color - gt) / (3 * H * W)

            def bwd():
                _C.rasterize_gaussians_backward(bg, act["means3D"], radii, E, act["scales"], act["rotations"], 1.0, E, cam.viewmatrix, cam.projmatrix,
                                                cam.tanfovx, cam.tanfovy, dLc, dLd, act["shs"], 3, cam.campos, geom, R, binb, img, False)
        else:
            import ref_harness as rh
            L = rh.rast(); p = rh._p
            col = torch.zeros(3, H, W, device=device); dep = torch.zeros(1, H, W, device=device)
            rad = torch.zeros(P, dtype=torch.int32, device=device)

            def fwd():
                col.zero_(); dep.zero_(); rad.zero_()
                st["R"] = L.ref_rast_forward(P, 3, 16, p(bg), W, H, p(act["means3D"]), p(act["shs"]), None, p(act["opacities"]), p(act["scales"]), 1.0,
                                             p(act["rotations"]), None, p(cam.viewmatrix), p(cam.projmatrix), p(cam.campos), cam.tanfovx, cam.tanfovy, 0,
                                             p(col), p(dep), p(rad), 0)
            fwd()
            R = st["R"]
            dLc = torch.sign(col - gt) / (3 * H * W)

            def bwd():
                z = lambda *s: torch.zeros(*s, device=device)
                g = [z(P, 3), z(P, 2, 2), z(P, 1), z(P, 3), z(P, 1), z(P, 3), z(P, 6), z(P, 16, 3), z(P, 3), z(P, 4)]
                L.ref_rast_backward(P, 3, 16, R, p(bg), W, H, p(act["means3D"]), p(act["shs"]), None, p(act["scales"]), 1.0, p(act["rotations"]), None,
                                    p(cam.viewmatrix), p(cam.projmatrix), p(cam.campos), cam.tanfovx, cam.tanfovy, p(rad), p(dLc), p(dLd),
                                    *[p(t) for t in g], 0)

        def timeit(fn, n=20, warm=5):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record(); torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        tf, tb = timeit(fwd), timeit(bwd)
        out[tag] = {"fwd_ms": round(tf, 4), "bwd_ms": round(tb, 4), "fwd_bwd_ms": round(tf + tb, 4), "fwd_bwd_per_s": 1e3 / (tf + tb),
                    "instances": int(R), "scene": f"scale_mu={mu}"}
        del raw, act
        torch.cuda.empty_cache()
    return out


# ---- stress (BASELINE.json config 5) -------------------------------------------------------------------
def stress_c5_block(args, device):
    """5M Gaussians at 3840x2160: `distCUDA2` initialisation (scene/gaussian_model.py:160-161), then training iterations of 2 views
    with a densification + pruning EVENT (GaussianModel.densify + prune through b200gs.densify: decision kernel + one gather)
    every 10 iterations, statistics accumulated every iteration (add_densification_stats, max_radii2D).  Reports the kNN time,
    the steady iteration time and every event's duration including the FIRST one (allocator growth included)."""
    from b200gs import engine, synthetic as syn
    from b200gs.knn import distCUDA2
    P, W, H, iters = 5_000_000, 3840, 2160, 31
    ev = lambda: torch.cuda.Event(enable_timing=True)
    raw = syn.make_gaussians(P, scale_mu=0.004, device="cpu")
    xyz = raw["xyz"].to(device)
    distCUDA2(xyz[:100000])                                    # library / allocator warm-up
    a, b = ev(), ev(); a.record()
    d2 = distCUDA2(xyz)
    b.record(); torch.cuda.synchronize()
    knn_ms = a.elapsed_time(b)
    raw["log_scale"] = torch.log(torch.sqrt(torch.clamp_min(d2, 1e-7)))[..., None].repeat(1, 3).cpu()
    torch.manual_seed(6666)
    model = engine.GaussianState({k: v.to(device) for k, v in raw.items()}, hyper=engine.default_hyper()).to(device)
    with torch.no_grad():
        model._deformation.deformation_net.set_aabb(xyz.max(0).values.tolist(), xyz.min(0).values.tolist())
    model.training_setup()
    model.densification_setup(percent_dense=0.01)
    h = engine.default_hyper()
    tr = engine.ViewParallelTrainer(model, torch.zeros(3, device=device), stage="fine",
                                    regulation=(h.time_smoothness_weight, h.l1_time_planes, h.plane_tv_weight))
    cams = syn.orbit_cameras(2, W, H, device=device)
    g = torch.Generator().manual_seed(99)
    gts = [(torch.rand(H, W, 3, generator=g) * 255.999).to(torch.uint8).to(device) for _ in cams]
    extent = 1.0
    step_ms, events = [], []
    n0 = P
    for it in range(1, iters + 1):
        a, b = ev(), ev(); a.record()
        loss = tr.step(cams, gts)
        with torch.no_grad():                                   # train_4DGS.py:264-267
            vis = tr.max_radii > 0
            model.max_radii2D = torch.maximum(model.max_radii2D, tr.max_radii.to(torch.float32))
            model.add_densification_stats(tr.viewspace_grad, vis)
        b.record()
        if it % 10 == 0:
            c, d = ev(), ev(); c.record()
            with torch.no_grad():
                before = model._xyz.shape[0]
                model.densify(0.0002, 0.005, extent, None)
                mid = model._xyz.shape[0]
                model.prune(0.0002, 0.005, extent, None)
            tr.rebuild()
            d.record(); torch.cuda.synchronize()
            events.append({"iteration": it, "ms": round(c.elapsed_time(d), 3), "points_before": before, "after_densify": mid, "after_prune": int(model._xyz.shape[0])})
        torch.cuda.synchronize()
        if not bool(torch.isfinite(loss).all()):
            raise RuntimeError("C5: non-finite loss")
        step_ms.append(a.elapsed_time(b))
    quiet = sorted(x for i, x in enumerate(step_ms) if i >= 2)          # median over every iteration after the two warm-up ones
    steady = quiet[len(quiet) // 2]
    out = {"config": "C5: 5,000,000 Gaussians, 3840x2160, 2 views per iteration, densify + prune event every 10 iterations", "distCUDA2_ms": round(knn_ms, 2),
           "iteration_ms_median": round(steady, 2), "iteration_ms_max_after_warmup": round(quiet[-1], 2), "view_iters_per_s": 2e3 / steady, "iteration_ms_all": [round(x, 1) for x in step_ms], "events": events,
           "max_memory_gib": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1), "reserved_gib": round(torch.cuda.memory_reserved() / 2 ** 30, 1),
           "cuda_mallocs": int(torch.cuda.memory_stats().get("num_device_alloc", 0)), "points_final": int(model._xyz.shape[0])}
    del tr, model
    torch.cuda.empty_cache()
    return out


# ---- the reference's own scripts through the launcher --------------------------------------------------
def launcher_path_block(args):
    """The boundary on hardware: the reference's UNCHANGED train_4DGS.py (baseline/_ref, installed by tools/install_reference.sh
    where /root/reference exists) run by `python -m b200gs.launcher` on the synthetic stage-1 stand-in (tools/make_synthetic_mom.py):
    210k initial Gaussians, 320x192, batch_size 2, 40 coarse + 120 fine iterations with densification and pruning.  iters/s is
    measured between the first and the last optimizer.step() of the run (so it includes everything the script does per
    iteration: its Python, the loss, densify / prune, tqdm), not the process start-up or data loading."""
    import re
    import shutil
    import tempfile
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "scene")):
        return {"unavailable": "baseline/_ref not installed"}
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_synthetic_mom as mm
    tmp = tempfile.mkdtemp(prefix="b200gs_launcher_")
    try:
        out = os.path.join(tmp, "scene")
        mm.write(out, points=210000, width=320, height=192, views=5, video_frames=60)
        cfg = mm.write_config(os.path.join(tmp, "short.py"), coarse_iterations=40, iterations=120, batch_size=2)
        env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "iclr2025_3d-mom_b200") + os.pathsep + os.environ.get("PYTHONPATH", ""),
                   B200GS_LAUNCHER_LOG="1")
        for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
            env.pop(k, None)
        runs = []
        for rep in range(3):          # a 159-iteration run lasts 1-2 s: one stray stall moves it by tens of percent (88-165 seen), so the median of 3
            t0 = time.perf_counter()
            r = subprocess.run([sys.executable, "-m", "b200gs.launcher", "--reference", ref, "train_4DGS.py", "--input_dir", out, "--configs", cfg,
                                "--expname", "synthetic", "--model_path", out, "--port", str(6124 + rep), "--save_iterations", "120",
                                "--test_iterations", "100000", "--video_iterations", "100000", "--quiet"],
                               cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
            wall = time.perf_counter() - t0
            m = re.search(r"\[b200gs\] launcher summary: (.*)", r.stdout + r.stderr)
            if r.returncode != 0 or not m:
                return {"failed": (r.stdout + r.stderr)[-600:]}
            summary = dict(kv.split("=") for kv in m.group(1).split())
            runs.append((float(summary["iters_per_s"]), wall, summary))
        runs.sort(key=lambda t: t[0])
        ips, wall, summary = runs[len(runs) // 2]
        return {"script": "train_4DGS.py (unchanged, baseline/_ref) via b200gs.launcher", "iters_per_s": ips,
                "iters_per_s_runs": [round(t[0], 1) for t in runs], "how": "median of 3 process runs",
                "view_iters_per_s": 2 * ips, "iterations": int(summary["adam_steps"]), "batch_size": 2,
                "points_initial": 210000, "image": "320x192", "process_wall_s": round(wall, 2),
                "densify_cat_events": int(summary["densify_cat_events"]), "prune_events": int(summary["prune_events"]),
                "time_row_forward_calls": int(summary["time_row_forward_calls"]),
                "spatial_product_evaluations": int(summary["spatial_product_evaluations"])}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


# ---- cpu baselines ---------------------------------------------------------------------------------
def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def cpu_c1(args):
    """BASELINE.json config 1 exactly as SURVEY.md 8(d) words it: the reference's PyTorch path on CPU tensors -- deform_network
    forward (effective config: 2 levels, T = 50, 64 features) + eval_sh degree 3 + clamp + cov3D (R S)(R S)^T + projection --
    200k synthetic Gaussians, 512x512 camera, one timestep, all host threads, 3 warm-up + 10 timed repetitions, median.
    Runs the pinned restatements (oracle/field_torch.py, oracle/cpu_path_torch.py): the reference tree does not exist here."""
    import statistics
    from b200gs import engine, synthetic as syn
    from b200gs.field import deform_network
    from oracle import cpu_path_torch as cp
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = 200_000
    raw = syn.make_gaussians(P, scale_mu=args.scale_mu, device="cpu")
    cam = syn.make_camera(512, 512)
    torch.manual_seed(6666)
    net = deform_network(engine.default_hyper())
    sd = {k: v.detach().clone().contiguous() for k, v in net.state_dict().items()}

    def once():
        t0 = time.perf_counter()
        with torch.no_grad():
            cp.c1_forward(sd, 2, raw["xyz"], raw["log_scale"], raw["rot"], raw["opacity_logit"], raw["shs"], raw["scene_flow"], 0.5, 3,
                          cam.viewmatrix, cam.projmatrix, cam.campos)
        return time.perf_counter() - t0
    first = once()
    warm, timed = (3, 10) if first < 1.5 else (1, 3)          # keep the leg inside ~30 s on a slow host
    for _ in range(warm - 1):
        once()
    ts = [once() for _ in range(timed)]
    med = statistics.median(ts)
    return {"config": "C1: HexPlane deformation + SH eval + projection forward, 200000 Gaussians, 512x512, 1 timestep", "seconds_median": med,
            "forwards_per_s": 1.0 / med, "warmup": warm, "timed": timed, "cores": cores, "cpu": _cpu_model(), "kind": "port",
            "seconds_all": [round(t, 4) for t in ts]}


def cpu_baseline(args, raw, cam):
    """CPU port of ONE view-iteration of the benchmarked workload (field fwd/bwd in torch on CPU tensors, rasterizer fwd/bwd in
    oracle/raster_cpu.c with OpenMP, Adam in C) on the host cores, on a bounded sample (--cpu-points Gaussians, image scaled with
    them), 1 warm-up + 2 timed repetitions (median), scaled linearly to the full workload.  Plus config 1 (`c1`)."""
    import statistics
    import numpy as np
    from b200gs import engine
    from oracle import field_torch, raster_cpu as rc
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    P = args.cpu_points or min(args.points, 200_000)
    frac = P / args.points
    W = max(16, int(round(args.width * frac ** 0.5 / 16)) * 16); H = max(16, int(round(args.height * frac ** 0.5 / 16)) * 16)
    from b200gs import synthetic as syn
    camc = syn.make_camera(W, H)
    sub = {k: v[:P].clone() for k, v in raw.items()}
    torch.manual_seed(6666)
    hyper = engine.default_hyper()
    from b200gs.field import deform_network
    net = deform_network(hyper)                   # reference-initialised field parameters, CPU tensors only
    gt = np.random.default_rng(0).random((3, H, W), dtype=np.float32)
    inst = [0]

    def once():
        sd = {k: v.detach().clone().contiguous().requires_grad_(v.dtype.is_floating_point and "poc" not in k and not k.endswith("aabb"))
              for k, v in net.state_dict().items()}
        xyz = sub["xyz"].clone().requires_grad_(True); scl = sub["log_scale"].clone().requires_grad_(True)
        rot = sub["rot"].clone().requires_grad_(True); opa = sub["opacity_logit"].clone().requires_grad_(True)
        shs = sub["shs"].clone().requires_grad_(True)
        t0 = time.perf_counter()
        tt = torch.full((P, 1), 0.5)
        pts, sc, rt, op, sh = field_torch.deform_forward(sd, 2, xyz, scl, rot, opa, shs, tt, sub["scene_flow"], 3, 1)
        a_sc, a_rt, a_op = torch.exp(sc), torch.nn.functional.normalize(rt), torch.sigmoid(op)
        s = rc.forward(pts.detach().numpy(), a_op.detach().numpy(), camc.viewmatrix.numpy(), camc.projmatrix.numpy(), camc.campos.numpy(),
                       W, H, camc.tanfovx, camc.tanfovy, np.zeros(3, np.float32), shs=sh.detach().numpy(), scales=a_sc.detach().numpy(),
                       rots=a_rt.detach().numpy())
        dL = np.sign(s["color"] - gt).astype(np.float32) / (3 * H * W)
        g = rc.backward(s, dL, np.zeros((1, H, W), np.float32))
        torch.autograd.backward([pts, a_sc, a_rt, a_op, sh],
                                [torch.from_numpy(g["means3D"]), torch.from_numpy(g["scales"]), torch.from_numpy(g["rotations"]),
                                 torch.from_numpy(g["opacity"]).reshape(P, 1), torch.from_numpy(g["sh"])])
        for q in [xyz, scl, rot, opa, shs] + [v for v in sd.values() if v.requires_grad and v.grad is not None]:
            pn = q.detach().numpy(); m = np.zeros_like(pn); v = np.zeros_like(pn)
            rc.adam_step(pn, q.grad.numpy().copy(), m, v, 1e-3, 1)
        inst[0] = int(s["R"])
        return time.perf_counter() - t0
    once()
    ts = [once(), once()]
    dt = statistics.median(ts)
    res = {"value": (1.0 / dt) * frac, "unit": "view-iters/s", "cores": cores, "kind": "port", "cpu": _cpu_model(),
           "sample": f"1 view-iteration (field fwd/bwd + raster fwd/bwd + Adam) at {P} Gaussians, {W}x{H}, 1 warm-up + 2 timed, median {dt:.2f} s, "
                     f"scaled by {frac:.3f} to the {args.points}-Gaussian {args.width}x{args.height} workload",
           "measured_seconds": dt, "instances": inst[0]}
    try:
        res["c1"] = cpu_c1(args)
    except Exception as ex:
        res["c1"] = {"failed": f"{type(ex).__name__}: {ex}"}
    return res


# ---------------------------------------------------------------------------------------------
def main():
    import contextlib
    # library chatter (Python prints AND C-level writes such as NCCL's version banner) goes to stderr;
    # the original stdout carries ONE JSON line
    sys.stdout.flush()
    real_fd = os.dup(1)
    os.dup2(2, 1)
    try:
        with contextlib.redirect_stdout(sys.stderr):
            line = _main()
    finally:
        sys.stdout.flush()
        os.dup2(real_fd, 1)
    if line is not None:
        os.write(real_fd, (line + "\n").encode())
    os.close(real_fd)


PHASES = ("preprocess_fwd", "depth_sort", "emit_instances", "tile_sort", "tile_ranges", "composite_fwd", "composite_bwd", "preprocess_bwd")


def read_phases():
    import ctypes
    from b200gs import _lib
    L = _lib.lib()
    L.b200gs_profile_read.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_float)]
    out = {}
    for name in PHASES:
        n, ms = ctypes.c_int(0), ctypes.c_float(0.0)
        if L.b200gs_profile_read(name.encode(), ctypes.byref(n), ctypes.byref(ms)) == 0 and n.value > 0:
            out[name] = {"calls": n.value, "ms_total": ms.value, "ms_avg": ms.value / n.value}
    return out


class no_gc:
    """Python's cyclic collector paused for a timed loop (collected once before it), both arms: the host waits for the GPU once
    per view (the instance-count read-back), so it is never more than a view ahead and a 10-20 ms generation-2 pause of the
    launching thread lands in the step time as is (seen as one slow step in ten).  Long training loops do the same."""

    def __enter__(self):
        import gc
        gc.collect()
        self.was = gc.isenabled()
        gc.disable()

    def __exit__(self, *exc):
        import gc
        if self.was:
            gc.enable()


def run_steps(trainer, cams, gts, n_global, steps, barrier, max_over_ranks):
    """K timed steps; returns (device ms, max over ranks; the loss tensor the last step returned, None if K = 0)."""
    loss = None
    with no_gc():
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = trainer.step(cams, gts, global_batch=n_global)
        e1.record()
        barrier()
    return max_over_ranks(e0.elapsed_time(e1)), loss


DUMP_ROWS = 65536           # Gaussians sampled (fixed seed) from each per-Gaussian tensor by dump_outputs
DUMP_LIMIT = 64 << 20       # bytes


def dump_outputs(out_dir, model, trainer, loss):
    """What one training step hands its caller, after the last timed step: the loss of the global batch (the sum over ranks of
    what each rank's step returned), every trainable parameter
    as the optimiser left it (grid planes in logical NCHW order) and the densification statistics the step accumulated
    (viewspace_grad, max_radii).  Per-Gaussian tensors are sampled to DUMP_ROWS rows chosen with a fixed seed, the rest are
    written whole; float32, except the loss (float64).  Same arguments, same inputs: two builds compare file by file."""
    import numpy as np
    if loss is None:
        raise SystemExit("--dump-outputs needs at least one timed step (--steps >= 1)")
    os.makedirs(out_dir, exist_ok=True)
    P = model._xyz.shape[0]
    rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(P, min(P, DUMP_ROWS), replace=False)))
    trainable = {id(p) for p in trainer.trainable}
    tensors = [(n, p) for n, p in model.named_parameters() if id(p) in trainable]
    tensors += [("viewspace_grad", trainer.viewspace_grad), ("max_radii", trainer.max_radii)]
    arrays = {"loss": np.array([float(loss)], dtype=np.float64)}
    for n, t in tensors:
        t = t.detach()
        if t.dim() > 0 and t.shape[0] == P:
            t = t[rows.to(t.device)]
        arrays[n] = t.float().contiguous().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


def run_steps_e2e(trainer, cams, host_images, n_global, steps, device, barrier, max_over_ranks, impl, warm=2):
    """Ground truth in pinned host memory, uploaded every step inside the timed region; loss read back every step.
    `warm` untimed steps through the SAME path first (both arms): the first end-to-end steps allocate the upload slots and settle
    the caching allocator after the instrumented pass that precedes them.  Returns (device ms, wall s, last loss, slowest step ms)."""
    from b200gs import engine
    last = None
    step_wall = []
    gc_pause = no_gc()
    gc_pause.__enter__()
    if impl == "b200":
        feeder = engine.HostImageFeeder(host_images, device)
        ring = engine.LossRing(depth=4)
        lag = 1 if len(cams) > 2 else 2
        feeder.prefetch()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = None
        for k in range(-warm, steps):
            if k == 0:
                for back in range(min(lag, ring.n) - 1, -1, -1):      # drain the warm-up's losses: the timed region starts empty
                    ring.read(lag=back)
                barrier()
                t_wall = time.perf_counter()
                f0.record()
            t_step = time.perf_counter()
            g = feeder.take()
            if k + 1 < steps:
                feeder.prefetch()                      # next step's upload overlaps this step
            loss = trainer.step(cams, g, global_batch=n_global)
            feeder.release()
            ring.push(loss)
            # every step's loss is read on the host, `lag` steps after it was queued: one step late while a step is long (N <= 4),
            # two when a rank's step is one or two views (5-7 ms) and the host needs that much queue depth to hide its own jitter
            v = ring.read(lag=lag)
            last = v if v is not None else last
            if k >= 0:
                step_wall.append(time.perf_counter() - t_step)
        for back in range(min(lag, steps) - 1, -1, -1):            # drain: the last `lag` losses
            v = ring.read(lag=back)
            last = v if v is not None else last
    else:
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = None
        for k in range(-warm, steps):                  # what train_4DGS.py:194,236 does: blocking float upload, loss.item() per step
            if k == 0:
                barrier()
                t_wall = time.perf_counter()
                f0.record()
            t_step = time.perf_counter()
            g_step = [g.to(device, non_blocking=True) for g in host_images]
            last = float(trainer.step(cams, g_step, global_batch=n_global))
            if k >= 0:
                step_wall.append(time.perf_counter() - t_step)
    f1.record()
    barrier()
    gc_pause.__exit__(None, None, None)
    return max_over_ranks(f0.elapsed_time(f1)), time.perf_counter() - t_wall, last, max(step_wall) * 1e3 if step_wall else 0.0


def _main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    impl = args.impl
    if impl == "reference-cpu":
        if rank != 0:
            return None
        from b200gs import synthetic as syn
        raw = syn.make_gaussians(args.points, scale_mu=args.scale_mu, device="cpu")
        cb = cpu_baseline(args, raw, None)
        return json.dumps({"impl": "reference", "metric": "train_iters_per_s", "value": cb["value"], "unit": "view-iters/s",
                           "n_gpus": 0, "steps": 1, "warmup": 0, "higher_is_better": True, "cpu_baseline": cb,
                           "e2e": {"value": cb["value"], "unit": "view-iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    launched_world = world
    if impl == "reference" and world > 1:
        # the reference has no multi-GPU path (INTEGRATION.md section 5): under torchrun rank 0 alone runs it, on one GPU,
        # and prints the line; the other ranks leave without work
        if rank != 0:
            return None
        world = 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)
    if args.global_batch % world != 0:
        raise SystemExit(f"--global-batch {args.global_batch} does not divide over {world} ranks")
    args.global_views = args.global_batch          # strong scaling: the batch BASELINE.json names, sharded over the ranks
    raw, cams, gts_host, n_global = build_scene(args, device, world, rank, impl)
    host_u8 = build_scene.last_u8
    if impl == "b200":
        model, trainer = make_b200_trainer(args, raw, device, world, rank)
    else:
        model, trainer = make_reference_trainer(args, raw, device, world, rank)
        if trainer is None:
            if rank == 0:
                return json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libref_rast.so missing (run oracle/build_ref.sh where /root/reference exists)"})
            return None
    # device-resident inputs of the `value` measurement: our arm keeps the dataset's uint8 images, the reference arm the float
    # tensors its loss needs
    gts_dev = [g.to(device, non_blocking=True) for g in (host_u8 if impl == "b200" else gts_host)]
    V = len(cams)
    pairs_per_view = None
    if impl == "b200":
        # evaluated (pixel, Gaussian) pairs = sum of n_contrib (SURVEY.md 8d), counted once, outside the timed region
        from b200gs import engine as _eng
        from b200gs.rasterizer import _C as _rc
        with torch.no_grad():
            _eng.render(cams[0], model, torch.zeros(3, device=device), stage="fine")
        try:
            sv = _eng.LAST_RASTER_STATE
            nc = _rc.export_state("n_contrib", args.points, sv[0], args.width, args.height, sv[1], sv[2], sv[3])
            pairs_per_view = int(nc.view(torch.int32).to(torch.int64).sum())
            instances = int(sv[0])
        except Exception:
            pairs_per_view, instances = None, None

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t[0])
        return ms

    # Per-entry-point device timing (CUDA events on the launching stream) is taken INSIDE the timed steps:
    # our arm through b200gs._lib.CallTimer + the library's phase timing, the reference arm for its optimiser step only.
    adam_ms = []
    opt_step = model.optimizer.step
    if impl != "b200":
        def timed_opt_step(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = opt_step(*a, **k); e1.record()
            adam_ms.append((e0, e1))
            return r
        model.optimizer.step = timed_opt_step

    W_ = max(args.warmup, 3)
    # (N > 1: three more untimed steps -- NCCL sets up its channels / algorithms for the two message sizes lazily, on two
    #  streams, and a straggling rank in the first timed steps showed up as a 15 % slower N = 4 line once)
    for _ in range(W_ + (3 if world > 1 else 0)):
        trainer.step(cams, gts_dev, global_batch=n_global)
    adam_ms.clear()
    timeline = None
    with ClockSampler(local, enabled=(rank == 0)) as clk:
        # headline: EXACTLY K un-instrumented steps between barriers, device time, max over ranks
        ms, last_loss = run_steps(trainer, cams, gts_dev, n_global, args.steps, barrier, max_over_ranks)
        if args.dump_outputs:
            if world > 1 and last_loss is not None:      # each rank's step returns its LOCAL share of the batch loss
                import torch.distributed as dist
                last_loss = last_loss.detach().clone()
                dist.all_reduce(last_loss)
            if rank == 0:
                dump_outputs(args.dump_outputs, model, trainer, last_loss)
        # the same K steps again with every entry point / rasterizer phase bracketed by CUDA events: the per-kernel durations
        # of the `kernels` table and the roofline (the ~150 extra event records per step make this pass a few per cent slower)
        calls, phases = {}, {}
        if impl == "b200":
            from b200gs import _lib as _b200lib
            # (with the views serialised on ONE stream: under view pipelining a kernel shares the SMs with the other stream's
            #  forward and its event-to-event time is no longer its own; `ms_per_step_serial_instrumented` is this pass)
            piped, trainer.pipeline_views = trainer.pipeline_views, False
            with _b200lib.CallTimer() as timer:
                _b200lib.lib().b200gs_profile_enable(1)
                ms_instr, _ = run_steps(trainer, cams, gts_dev, n_global, args.steps, barrier, max_over_ranks)
                calls = timer.summary()
                phases = read_phases()
                _b200lib.lib().b200gs_profile_enable(0)
            trainer.pipeline_views = piped
            adam_t = calls.get("b200gs_adam_multi", {}).get("ms_avg", 0.0)
        else:
            ms_instr = ms
            adam_t = sum(a.elapsed_time(b) for a, b in adam_ms) / max(len(adam_ms), 1)
        ms_e2e, wall_e2e, last, e2e_slowest = run_steps_e2e(trainer, cams, host_u8 if impl == "b200" else gts_host, n_global, args.steps,
                                                            device, barrier, max_over_ranks, impl)
        if impl == "b200":
            # where one step's time goes: CUDA events around its phases (main stream + the SH side stream), one extra step
            trainer.timeline = {}
            trainer.step(cams, gts_dev, global_batch=n_global)
            torch.cuda.synchronize()
            tl, trainer.timeline = trainer.timeline, None
            def span(a, b):
                return round(tl[a].elapsed_time(tl[b]), 4) if a in tl and b in tl else None
            timeline = {"views_ms": span("step_start", "views_done"), "deferred_field_backward_ms": span("views_done", "field_done"),
                        "arena_allreduce_ms": span("field_done", "arena_reduced"), "regulariser_adam_ms": span("arena_reduced", "adam_done"),
                        "join_sh_side_stream_ms": span("adam_done", "step_end"), "step_ms": span("step_start", "step_end"),
                        "sh_side_stream": {"start_after_step_start_ms": span("step_start", "sh_tail_start"),
                                           "allreduce_sh_and_radii_ms": span("sh_tail_start", "sh_reduced"),
                                           "adam_sh_ms": span("sh_reduced", "sh_tail_end"),
                                           "end_after_step_start_ms": span("step_start", "sh_tail_end")}}
    if impl != "b200":
        model.optimizer.step = opt_step

    # ---- weak-scaling block (N > 1): 8 views per GPU, global batch 8 N ----
    weak = None
    if world > 1 and impl == "b200" and not args.no_weak:
        from b200gs import synthetic as syn
        nw = args.views_per_gpu * world
        cams_w = syn.orbit_cameras(nw, args.width, args.height, device=device)[rank::world]
        g = torch.Generator().manual_seed(4321 + rank)
        host_w = [(torch.rand(args.height, args.width, 3, generator=g) * 255.999).to(torch.uint8).pin_memory() for _ in cams_w]
        dev_w = [h.to(device) for h in host_w]
        for _ in range(2):
            trainer.step(cams_w, dev_w, global_batch=nw)
        ms_w, _ = run_steps(trainer, cams_w, dev_w, nw, args.steps, barrier, max_over_ranks)
        ms_we, _, _, _ = run_steps_e2e(trainer, cams_w, host_w, nw, args.steps, device, barrier, max_over_ranks, impl)
        weak = {"scaling": "weak", "views_per_gpu": args.views_per_gpu, "global_batch": nw, "value": nw * args.steps / (ms_w / 1e3),
                "unit": "view-iters/s", "ms_per_step": ms_w / args.steps, "e2e_value": nw * args.steps / (ms_we / 1e3)}
        del host_w, dev_w

    render = None
    render_note = None
    if args.render_frames > 0:
        try:
            render = render_block(args, model, device, world, rank, impl, ref_render=None if impl == "b200" else trainer.render_fn)
        except Exception as ex:                      # the side measurement must not take the headline down: fall back to per-frame passes
            if impl != "b200" or args.no_shared_spatial:
                raise
            render_note = f"shared spatial product failed ({type(ex).__name__}: {ex}); per-frame six-plane passes measured instead"
            args.no_shared_spatial = True
            from b200gs import field as _field
            _field.drop_shared()
            render = render_block(args, model, device, world, rank, impl, ref_render=None)
    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return None

    views_total = n_global * args.steps
    value = views_total / (ms / 1e3)
    e2e_value = views_total / (ms_e2e / 1e3)
    pk, pk_kind = peaks()
    hbm = pk.get("hbm_gbs")
    n_params = sum(p.numel() for p in trainer.trainable)
    n_sh = sum(p.numel() for p in getattr(trainer, "sh_params", []))
    P_, F_ = args.points, 64
    plane_params = sum(p.numel() for n, p in model.named_parameters() if ".grids." in n)
    R_ = instances if impl == "b200" and instances else 0
    tiles = ((args.width + 15) // 16) * ((args.height + 15) // 16)
    tile_bits = max(1, (tiles - 1).bit_length())
    tile_passes = (tile_bits + 7) // 8
    fp32_peak = 148 * 128 * 1.965e9                 # lane-instructions per second (SURVEY.md 8d)
    # algorithmic HBM bytes per launch (DESIGN.md section 3; SURVEY.md 8d): what each kernel must move when every
    # re-used operand (planes, weights) stays on chip
    entry_models = {
        "b200gs_adam_multi": ("adam_multi_kernel", 28.0 * (n_params - n_sh)),
        "b200gs_adam_sh": ("adam_sh_kernel", 28.0 * n_sh),
        "b200gs_hexplane_forward": ("hexplane_fwd_kernel", P_ * (12 + 4 + 4 * F_)),
        "b200gs_hexplane_backward": ("hexplane_bwd_kernel", P_ * (12 + 4 + 4 * F_ + 12) + 4 * plane_params),
        "b200gs_hexplane_forward_masked": ("hexplane_fwd_kernel (spatial planes, once per step)", P_ * (12 + 4 + 4 * F_)),
        "b200gs_hexplane_backward_masked": ("hexplane_bwd_kernel (spatial planes, once per step)", P_ * (12 + 4 + 4 * F_ + 12) + 4 * plane_params),
        "b200gs_hexplane_time_forward": ("hexplane_time_fwd2_kernel", P_ * (12 + 4 * F_ + 4 * F_)),
        "b200gs_hexplane_time_backward": ("hexplane_time_bwd2_kernel", P_ * (12 + 4 * F_ + 4 * F_ + 8 * F_ + 12)),
        "b200gs_deform_mlp_forward": ("deform_mlp_fwd_tc5v2_kernel", P_ * (4 * F_ + 52 + 4 * 4 * 64 + 40)),
        "b200gs_deform_mlp_backward": ("deform_mlp_bwd_tc5_kernel", P_ * (4 * 4 * 64 + 4 * F_ + 40 + 4 * F_)),
        "b200gs_activations_forward": ("activations_fwd_kernel", P_ * 64),
        "b200gs_activations_backward": ("activations_bwd_kernel", P_ * 96),
        "b200gs_l1_loss_fwd_bwd": ("l1_fwd_bwd_kernel", 12 * 3 * args.width * args.height),
        "b200gs_l1_loss_fwd_bwd_u8": ("l1_fwd_bwd_u8_kernel", (4 + 1 + 4) * 3 * args.width * args.height),
        "b200gs_hexplane_regulation": ("hexplane_regulation_kernel", 8.0 * plane_params),
    }
    phase_models = {      # SURVEY.md 8(d) formulas
        "preprocess_fwd": ("preprocess_fwd_kernel", "hbm", 311.0 * P_),
        "depth_sort": ("rs_histogram + rs_scan_hist + 4 x rs_onesweep_pass (32-bit depth keys + index)", "hbm", (4 + 4 * 16.0) * P_),
        "emit_instances": ("emit_instances_kernel", "hbm", 16.0 * P_ + 8.0 * R_),
        "tile_sort": (f"rs_histogram + rs_scan_hist + {tile_passes} x rs_onesweep_pass (tile id + Gaussian id)", "hbm", (4 + tile_passes * 16.0) * R_),
        "tile_ranges": ("tile_ranges_kernel", "hbm", 4.0 * R_ + 8.0 * tiles),
        "composite_fwd": ("composite_fwd_kernel", "fp32-issue", 30.0 * (pairs_per_view or 0)),
        "composite_bwd": ("composite_bwd2_kernel", "fp32-issue", 85.0 * (pairs_per_view or 0)),
        "preprocess_bwd": ("preprocess_bwd_kernel", "hbm", 622.0 * P_),
    }
    # the reference's own sort moves (8 + 24 * ceil((32 + bits) / 8)) B per instance (64-bit keys): for comparison
    ref_sort_bytes = (8 + 24 * ((32 + tile_bits + 7) // 8)) * R_
    traffic, traffic_src = ncu_traffic()
    kernels = []
    for name, c in sorted(calls.items(), key=lambda kv: -kv[1]["ms_total"]):
        row = {"entry": name, "calls": c["calls"], "ms_avg": round(c["ms_avg"], 4), "share_of_step": round(c["ms_total"] / ms_instr, 4)}
        if name in entry_models and c["ms_avg"] > 0:
            kname, nbytes = entry_models[name]
            gbs = nbytes / (c["ms_avg"] * 1e-3) / 1e9
            row.update({"kernel": kname, "bound": "hbm", "algorithmic_bytes_per_launch": nbytes, "achieved_gbs": round(gbs, 1),
                        "frac_of_measured_hbm_peak": round(gbs / hbm, 4)})
        kernels.append(row)
    for name, c in sorted(phases.items(), key=lambda kv: -kv[1]["ms_total"]):
        kname, bound, work = phase_models[name]
        row = {"phase": name, "kernel": kname, "calls": c["calls"], "ms_avg": round(c["ms_avg"], 4), "share_of_step": round(c["ms_total"] / ms_instr, 4),
               "bound": bound}
        if c["ms_avg"] > 0 and work > 0:
            if bound == "hbm":
                gbs = work / (c["ms_avg"] * 1e-3) / 1e9
                row.update({"algorithmic_bytes_per_launch": work, "achieved_gbs": round(gbs, 1), "frac_of_measured_hbm_peak": round(gbs / hbm, 4)})
            else:
                rate = work / (c["ms_avg"] * 1e-3)
                row.update({"pairs_per_launch": pairs_per_view, "lane_instr_per_pair_reference_cost_model": work / max(pairs_per_view, 1),
                            "achieved_lane_instr_per_s": rate, "frac_of_fp32_peak_on_reference_cost_model": round(rate / fp32_peak, 4)})
        kernels.append(row)
    single = [k for k in kernels if "frac_of_measured_hbm_peak" in k and ("phase" in k or not k["entry"].startswith("b200gs_rast_"))]
    single.sort(key=lambda k: -k["share_of_step"])
    dom = single[0] if single else None
    launches_per_step = None
    if impl == "b200":
        # kernels of libb200gs launched in the timed region, counted per entry point by CallTimer (KERNELS table)
        launches_per_step = sum(c["kernels"] for c in calls.values()) / args.steps
    vpg = n_global // world
    res = {
        "metric": "train_iters_per_s", "value": value, "unit": "view-iters/s", "n_gpus": world, "steps": args.steps,
        "warmup": W_, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"C3 train_4DGS fine-stage iteration: HexPlane deform + raster fwd/bwd + plane regulariser + Adam, {args.points} Gaussians, "
                               f"{args.width}x{args.height}, global batch {n_global} views per optimizer step over {world} GPU(s) ({vpg} per GPU)",
                   "scene": f"seeded synthetic, scale_mu={args.scale_mu}", "global_batch": n_global, "views_per_gpu": vpg,
                   "iters_per_s_at_batch": value / n_global,
                   "host": "python cyclic GC paused during the timed loops (collected before each), both arms",
                   "l2": "per-step working set (>= 236 MB of parameters + Adam state + 1M-splat records) exceeds the 126 MB L2",
                   "parallelism": f"view-parallel dp{world}"},
        "e2e": {"value": e2e_value, "unit": "view-iters/s",
                "h2d_bytes_per_step": V * 3 * args.height * args.width * (1 if impl == "b200" else 4),
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps, "wall_ms_per_step": wall_e2e * 1e3 / args.steps,
                "warmup_steps": 2, "slowest_step_wall_ms": e2e_slowest, "last_loss": last,
                "how": ("uint8 HWC ground truth (the dataset's own format) uploaded from pinned memory on a side stream one step ahead, converted "
                        "inside the L1 kernel; loss copied to a pinned ring every step and read one step late (two when a rank's step is one or two views)") if impl == "b200" else
                       "float32 CHW ground truth uploaded per step, float(loss) per step (train_4DGS.py:194, :236)"},
        "clocks": clk.summary(),
        "gpu_launches": int(round(launches_per_step * args.steps)) if launches_per_step else 0,
    }
    peak_src = pk_kind + " (MEASURED_PEAKS.json hbm_gbs)" if pk_kind == "measured" else "fallback 6650"
    if impl == "b200" and dom is not None:
        # the dominant kernel of the step by device time
        compulsory = 92.0 * P_ if "deform_mlp" in dom["kernel"] else None
        res["roofline"] = {"kernel": dom["kernel"], "bound": "hbm", "achieved": dom["achieved_gbs"], "peak": hbm, "unit": "GB/s",
                           "frac": dom["frac_of_measured_hbm_peak"], "traffic": traffic.get(dom["kernel"].split(" ")[0]),
                           "traffic_source": traffic_src, "peak_source": peak_src,
                           "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"], "ms_per_launch": dom["ms_avg"],
                           "share_of_step": dom["share_of_step"],
                           "note": ("algorithmic bytes = this kernel's interface (activation stash 1 KB + features + d_features + 40 B of upstream "
                                    "gradients per point); SURVEY.md 8(d)'s compulsory bytes for a fully fused HexPlane+MLP backward are 92 B/point "
                                    "(see compulsory_frac): the stash and the feature rows are design traffic") if compulsory else ""}
        if compulsory:
            res["roofline"]["compulsory_bytes_per_launch"] = compulsory
            res["roofline"]["compulsory_frac"] = round(compulsory / (dom["ms_avg"] * 1e-3) / 1e9 / hbm, 4)
        res["kernels"] = kernels
        res["kernels_pass_ms_per_step"] = ms_instr / args.steps
        res["kernels_pass"] = ("the per-kernel pass brackets every entry point with CUDA events and runs the views of a step one after the other "
                               "on one stream (the timed headline pipelines them over two), so each duration is the kernel's own")
        res["reference_sort_bytes_per_view"] = ref_sort_bytes
        if timeline:
            res["timeline"] = timeline
    else:
        adam_bytes = 28.0 * n_params
        adam_gbs = adam_bytes / (adam_t * 1e-3) / 1e9 if adam_t > 0 else None
        res["roofline"] = {"kernel": "torch foreach Adam", "bound": "hbm", "achieved": adam_gbs, "peak": hbm, "unit": "GB/s",
                           "frac": (adam_gbs / hbm) if adam_gbs else None, "traffic": None, "peak_source": peak_src,
                           "algorithmic_bytes_per_launch": adam_bytes, "ms_per_launch": adam_t, "params": n_params}
    if weak is not None:
        res["weak"] = weak
    if impl == "b200":
        # which kernel generations ran (include/b200gs.h: b200gs_set_option; environment B200GS_* overrides)
        try:
            from b200gs import _lib as _l
            res["config"]["kernel_options"] = {n: int(_l.lib().b200gs_get_option(n.encode()))
                                               for n in ("mlp_fwd_elect", "mlp_bwd_v2", "hexplane_time_fwd", "hexplane_time_bwd", "lookback_parallel", "composite_pairs", "sort_ballot_rank")}
            res["config"]["overlap_sh_reduce"] = bool(trainer.overlap_sh_reduce)
        except Exception as ex:              # informational only
            res["config"]["kernel_options"] = f"unavailable: {ex}"
    if render is not None:
        res["render"] = render
        res["config"]["render"] = (f"video rendering (config C4), 5 camera paths x {args.render_frames} frames with advancing time, frames sharded "
                                   "round-robin over ranks; fps = device time, e2e_fps = wall clock incl. to8b + D2H per frame"
                                   + ("" if impl != "b200" or args.no_shared_spatial else
                                      "; spatial HexPlane product evaluated once per path (engine.render_frames), time planes per frame"))
        if render_note:
            res["config"]["render_note"] = render_note
    if not args.no_raster_only:
        try:
            res["raster_only"] = raster_only_block(args, device, impl)
        except Exception as ex:
            res["raster_only"] = {"failed": f"{type(ex).__name__}: {ex}"}
    if impl == "b200" and world == 1 and not args.no_c5:
        trainer = model = None                              # free the C3 model before the 5M-Gaussian one is built
        torch.cuda.empty_cache()
        try:
            res["stress_c5"] = stress_c5_block(args, device)
        except Exception as ex:
            res["stress_c5"] = {"failed": f"{type(ex).__name__}: {ex}"}
    if impl == "b200" and world == 1 and not args.no_launcher_path:
        torch.cuda.empty_cache()
        try:
            res["launcher_path"] = launcher_path_block(args)
        except Exception as ex:
            res["launcher_path"] = {"failed": f"{type(ex).__name__}: {ex}"}
    if impl != "b200":
        res["impl"] = "reference"
        res["reference_stack"] = "reference CUDA rasterizer (oracle/_ref, unmodified) + PyTorch port of HexPlane/deformation + torch.optim.Adam, on GPU"
        if launched_world > 1:
            res["n_gpus"] = launched_world
            res["ranks_used"] = 1
            res["config"]["parallelism"] = f"single GPU (the reference has no multi-GPU path; launched with {launched_world} ranks, rank 0 ran)"
        # schema completeness: this arm is the reference's own implementation of the path, which is CUDA (it has no CPU
        # implementation); one host thread drives it. The CPU port is what `cpu_baseline` on the product line times.
        res["cpu_baseline"] = {"value": value, "unit": "view-iters/s", "cores": 1, "kind": "reference",
                               "sample": "the reference's own code path for this workload (its CUDA rasterizer from oracle/_ref + its PyTorch "
                                         "field + torch Adam) on the same GPU, full workload; host side single-threaded"}
    if not args.no_cpu_baseline and world == 1 and impl == "b200":
        try:
            res["cpu_baseline"] = cpu_baseline(args, raw, cams[0])
        except Exception as ex:          # the checker must never take the product line down
            res["cpu_baseline"] = {"value": None, "unit": "view-iters/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return json.dumps(res)


if __name__ == "__main__":
    main()
