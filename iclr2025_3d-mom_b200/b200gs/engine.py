"""Host-side hot loop: the model state, `render()` and the view-parallel training step.

This is the part of the reference's L2/L3 layers that the hot path needs, restated so that
bench.py, the tests and the multi-GPU trainer can drive the kernels without the reference
tree (which does not exist on the GPU box):
  * `GaussianState`  — the tensors and optimiser groups of scene/gaussian_model.py:55-70, :190-209
                       (same attribute names: _xyz, _features_dc, _features_rest, _scaling,
                       _rotation, _opacity, _scene_flow, _deformation; same 8 Adam groups / lrs)
  * `render()`       — gaussian_renderer/__init__.py:22-178 (settings, deformation in the fine
                       stage, exp / normalize / sigmoid activations, rasterizer call, result dict)
  * `ViewParallelTrainer` — train_4DGS.py:172-297 for a batch of views, with the batch sharded
                       over ranks: every rank renders its views, one flat NCCL all-reduce sums the
                       gradients (Gaussians | planes | MLP | screen-space xy), every rank takes
                       the identical fused Adam step (SURVEY.md §8e).
With the real reference tree on sys.path, train_4DGS.py / render_4DGS.py run unchanged through
b200gs.launcher instead (INTEGRATION.md).
"""
import math
import os
import types

import torch
import torch.nn as nn

from . import fusedops
from . import rasterizer as _rast
from .adam import FusedAdam
from .field import deform_network
from .rasterizer import GaussianRasterizationSettings, GaussianRasterizer


def default_hyper(multires=(1, 2), time_res=50):
    """ModelHiddenParams as train_4DGS.py sees them with its default config
    (arguments/__init__.py:75-106 overridden by arguments/dnerf/hellwarrior.py + dnerf_default.py)."""
    return types.SimpleNamespace(
        net_width=64, timebase_pe=4, defor_depth=0, posebase_pe=10, scale_rotation_pe=2, opacity_pe=2,
        timenet_width=64, timenet_output=32, bounds=1.6, plane_tv_weight=0.0001, time_smoothness_weight=0.01,
        l1_time_planes=0.0001, grid_pe=0,
        kplanes_config={'grid_dimensions': 2, 'input_coordinate_dim': 4, 'output_coordinate_dim': 32,
                        'resolution': [64, 64, 64, time_res]},
        multires=list(multires), no_dx=False, no_grid=False, no_ds=False, no_dr=False, no_do=True, no_dshs=True,
        empty_voxel=False, static_mlp=False, apply_rotation=False)


def default_opt():
    """OptimizationParams (arguments/__init__.py:110-151 + dnerf_default.py)."""
    return types.SimpleNamespace(
        position_lr_init=0.00016, position_lr_final=0.0000016, position_lr_delay_mult=0.01, position_lr_max_steps=20000,
        deformation_lr_init=0.00016, deformation_lr_final=0.0000016, deformation_lr_delay_mult=0.01,
        grid_lr_init=0.0016, grid_lr_final=0.000016, feature_lr=0.0025, opacity_lr=0.05, scaling_lr=0.005,
        rotation_lr=0.001, percent_dense=0.01, lambda_dssim=0.0)


def expon_lr(step, lr_init, lr_final, max_steps, lr_delay_steps=0, lr_delay_mult=1.0):
    """The reference's learning-rate schedule (utils/general_utils.py:35-68, get_expon_lr_func): log-linear interpolation from
    lr_init at step 0 to lr_final at max_steps, optionally eased in by a reverse-cosine delay. Python floats, like the
    reference (the optimiser reads `param_group['lr']` on the host)."""
    if step < 0 or (lr_init == 0.0 and lr_final == 0.0):
        return 0.0
    if lr_delay_steps > 0:
        delay_rate = lr_delay_mult + (1 - lr_delay_mult) * math.sin(0.5 * math.pi * min(max(step / lr_delay_steps, 0.0), 1.0))
    else:
        delay_rate = 1.0
    t = min(max(step / max_steps, 0.0), 1.0)
    return delay_rate * math.exp(math.log(lr_init) * (1 - t) + math.log(lr_final) * t)


class GaussianState(nn.Module):
    def __init__(self, raw, sh_degree=3, hyper=None, spatial_lr_scale=1.0):
        """raw: dict from b200gs.synthetic.make_gaussians (xyz, log_scale, rot, opacity_logit, shs, scene_flow)."""
        super().__init__()
        self.max_sh_degree = sh_degree
        self.active_sh_degree = sh_degree
        self.spatial_lr_scale = spatial_lr_scale
        self._xyz = nn.Parameter(raw["xyz"].clone())
        self._features_dc = nn.Parameter(raw["shs"][:, :1, :].clone().contiguous())
        self._features_rest = nn.Parameter(raw["shs"][:, 1:, :].clone().contiguous())
        self._scaling = nn.Parameter(raw["log_scale"].clone())
        self._rotation = nn.Parameter(raw["rot"].clone())
        self._opacity = nn.Parameter(raw["opacity_logit"].clone())
        self.register_buffer("_scene_flow", raw["scene_flow"].clone())
        self._deformation = deform_network(hyper or default_hyper())
        self.optimizer = None

    # accessors named as in scene/gaussian_model.py:117-147
    @property
    def get_xyz(self):
        return self._xyz

    @property
    def get_features(self):
        return torch.cat((self._features_dc, self._features_rest), dim=1)

    @property
    def get_flow(self):
        return self._scene_flow

    scaling_activation = staticmethod(torch.exp)
    opacity_activation = staticmethod(torch.sigmoid)
    rotation_activation = staticmethod(torch.nn.functional.normalize)

    def training_setup(self, opt=None):
        opt = opt or default_opt()
        s = self.spatial_lr_scale
        groups = [
            {'params': [self._xyz], 'lr': opt.position_lr_init * s, "name": "xyz"},
            {'params': list(self._deformation.get_mlp_parameters()), 'lr': opt.deformation_lr_init * s, "name": "deformation"},
            {'params': list(self._deformation.get_grid_parameters()), 'lr': opt.grid_lr_init * s, "name": "grid"},
            {'params': [self._features_dc], 'lr': opt.feature_lr, "name": "f_dc"},
            {'params': [self._features_rest], 'lr': opt.feature_lr / 20.0, "name": "f_rest"},
            {'params': [self._opacity], 'lr': opt.opacity_lr, "name": "opacity"},
            {'params': [self._scaling], 'lr': opt.scaling_lr, "name": "scaling"},
            {'params': [self._rotation], 'lr': opt.rotation_lr, "name": "rotation"}]
        self.optimizer = FusedAdam(groups, lr=0.0, eps=1e-15)
        self._lr_args = {"xyz": (opt.position_lr_init * s, opt.position_lr_final * s),
                         "deformation": (opt.deformation_lr_init * s, opt.deformation_lr_final * s),
                         "grid": (opt.grid_lr_init * s, opt.grid_lr_final * s)}
        self._lr_max_steps = opt.position_lr_max_steps
        return self.optimizer

    # ---- densification bookkeeping, names and semantics of scene/gaussian_model.py:190-196, :681-715 ----
    def densification_setup(self, percent_dense=0.01):
        N, dev = self._xyz.shape[0], self._xyz.device
        self.percent_dense = percent_dense
        self.xyz_gradient_accum = torch.zeros((N, 1), device=dev)
        self.denom = torch.zeros((N, 1), device=dev)
        self.max_radii2D = torch.zeros((N,), device=dev)
        self._deformation_accum = torch.zeros((N, 3), device=dev)
        self._deformation_table = torch.ones((N,), dtype=torch.bool, device=dev)
        if self.optimizer is not None:
            from . import densify as _d
            _d.warmup(self)                  # first-use costs and allocator growth paid here, not inside the first event

    def add_densification_stats(self, viewspace_point_tensor, update_filter):
        from . import densify as _d
        _d.add_densification_stats(self, viewspace_point_tensor, update_filter)

    def densify(self, max_grad, min_opacity, extent, max_screen_size, *a, **k):
        from . import densify as _d
        _d.densify(self, max_grad, min_opacity, extent, max_screen_size)

    def prune(self, max_grad, min_opacity, extent, max_screen_size):
        from . import densify as _d
        _d.prune(self, max_grad, min_opacity, extent, max_screen_size)

    def reset_opacity(self):
        from . import densify as _d
        _d.reset_opacity(self)

    # model files (scene/gaussian_model.py:321-360, 367-407): same bytes on disk, see b200gs/modelio.py
    def save_ply(self, path):
        from . import modelio
        modelio.save_ply(self, path)

    def load_ply(self, path):
        from . import modelio
        modelio.load_ply(self, path)

    def save_deformation(self, path):
        from . import modelio
        modelio.save_deformation(self, path)

    def load_model(self, path):
        from . import modelio
        modelio.load_model(self, path)

    def update_learning_rate(self, iteration):
        """scene/gaussian_model.py:284-298: per-iteration schedule of the xyz / grid / deformation groups (all three decay
        over position_lr_max_steps; the other groups keep their constant rates)."""
        for group in self.optimizer.param_groups:
            name = group["name"]
            key = "xyz" if name == "xyz" else ("grid" if "grid" in name else ("deformation" if name == "deformation" else None))
            if key is not None:
                lr_init, lr_final = self._lr_args[key]
                group["lr"] = expon_lr(iteration, lr_init, lr_final, self._lr_max_steps)


LAST_RASTER_STATE = None      # (R, geomBuffer, binningBuffer, imgBuffer) of the last no-grad render (bench.py counts pairs from it)


def render(cam, pc, bg_color, scaling_modifier=1.0, stage="fine", delta_scale=1, debug=False, shs=None, leaves=None):
    """gaussian_renderer/__init__.py:22-178 for a b200gs.synthetic.SynthCamera-like `cam`.
    `shs`: optional pre-concatenated [P,16,3] SH tensor standing in for `pc.get_features` (the trainer
    concatenates once per optimiser step instead of once per view; the values are identical).
    `leaves`: optional (xyz, opacity, scaling, rotation) leaf tensors standing in for the model's parameters (same storage,
    same .grad buffers: the trainer's per-stream aliases, see ViewParallelTrainer._alias_leaves)."""
    means3D = pc.get_xyz if leaves is None else leaves[0]
    screenspace_points = torch.zeros_like(means3D, requires_grad=True)
    settings = GaussianRasterizationSettings(
        image_height=int(cam.image_height), image_width=int(cam.image_width), tanfovx=cam.tanfovx, tanfovy=cam.tanfovy,
        bg=bg_color, scale_modifier=scaling_modifier, viewmatrix=cam.viewmatrix, projmatrix=cam.projmatrix,
        sh_degree=pc.active_sh_degree, campos=cam.campos, prefiltered=False, debug=debug)
    rasterizer = GaussianRasterizer(raster_settings=settings)
    opacity, scales, rotations = (pc._opacity, pc._scaling, pc._rotation) if leaves is None else leaves[1:]
    if shs is None:
        shs = pc.get_features
    if stage == "coarse":
        m3, sc, rt, op, sh = means3D, scales, rotations, opacity, shs
    else:
        # the reference repeats the camera's timestamp into a [P,1] tensor (gaussian_renderer/__init__.py:56); our field
        # takes the scalar itself (CUDA path only), which also tells its backward that the whole view shares one time
        time = float(cam.time) if means3D.is_cuda else torch.full((means3D.shape[0], 1), float(cam.time), device=means3D.device)
        m3, sc, rt, op, sh = pc._deformation(means3D, scales, rotations, opacity, shs, time, pc.get_flow,
                                             cam.frame_num, delta_scale)
    if sc.is_cuda:
        sc, rt, op = fusedops.activations(sc, rt, op)      # exp / F.normalize / sigmoid in one launch each way
    else:                                                   # CPU tensors only reach here from the gloo plumbing test
        sc = pc.scaling_activation(sc); rt = pc.rotation_activation(rt); op = pc.opacity_activation(op)
    image, radii, depth = rasterizer(means3D=m3, means2D=screenspace_points, shs=sh, colors_precomp=None,
                                     opacities=op, scales=sc, rotations=rt, cov3D_precomp=None)
    if not torch.is_grad_enabled():
        global LAST_RASTER_STATE
        LAST_RASTER_STATE = getattr(rasterizer, "last_state", None)
    return {"render": image, "viewspace_points": screenspace_points, "visibility_filter": radii > 0, "radii": radii,
            "depth": depth}


def render_frames(cams, pc, bg_color, stage="fine", streams=2, **kw):
    """render() for every camera of a sequence over ONE static model (render_4DGS.py:41-76), as a generator: in the fine
    stage the time-independent half of the HexPlane field is evaluated once for the whole sequence
    (field.shared_spatial_product) instead of once per frame.
    streams = 2 (GPU): consecutive frames alternate between two side streams, so that frame i+1's field + preprocess + depth
    sort run under frame i's binning and compositing (all latency-bound: a frame alone leaves most SMs idle, and the host waits
    once per frame for the instance count).  The caller's stream waits for a frame before it is yielded, so whatever the
    consumer queues (output.FrameStore.put, a loss) is ordered after it without knowing about the streams."""
    import contextlib
    from . import field as _field
    on_gpu = pc.get_xyz.is_cuda
    with contextlib.ExitStack() as stack:
        if stage == "fine" and on_gpu:
            with torch.no_grad():
                stack.enter_context(_field.shared_spatial_product(pc._deformation, pc._xyz))
        pool = None
        if on_gpu and streams and streams > 1:
            cur = torch.cuda.current_stream()
            pool = _frame_streams(pc.get_xyz.device, int(streams))
            for st in pool:
                st.wait_stream(cur)            # parameters and the spatial product are ready
        for i, cam in enumerate(cams):
            if pool is None:
                with torch.no_grad():          # per frame, not across the yield: the consumer keeps its own grad mode
                    out = render(cam, pc, bg_color, stage=stage, **kw)
            else:
                st = pool[i % len(pool)]
                with torch.no_grad(), torch.cuda.stream(st):
                    out = render(cam, pc, bg_color, stage=stage, **kw)
                    done = torch.cuda.Event()
                    done.record(st)
                cur = torch.cuda.current_stream()
                cur.wait_event(done)
                for v in out.values():         # allocated on the side stream, consumed on the caller's
                    if torch.is_tensor(v) and v.is_cuda:
                        v.record_stream(cur)
            yield out
        if pool is not None:                   # nothing of the sequence may outlive the shared product it reads
            cur = torch.cuda.current_stream()
            for st in pool:
                cur.wait_stream(st)


_FRAME_STREAMS = {}


def _frame_streams(device, n):
    key = (torch.device(device).index, n)
    if key not in _FRAME_STREAMS:
        _FRAME_STREAMS[key] = [torch.cuda.Stream(device=device) for _ in range(n)]
    return _FRAME_STREAMS[key]


class HostImageFeeder:
    """Ground-truth images that live in HOST memory the way the dataset holds them (PIL -> uint8 [H,W,3],
    scene/dataset_readers.py:1041-1057; the reference uploads a float32 copy per view, train_4DGS.py:194): `take()` returns
    this step's images on the device, `prefetch()` queues the next step's host->device copies on a side stream so that they
    overlap the current step; the L1 kernel converts u8 -> float on the device (fusedops.l1_loss_and_grad).  3 bytes per pixel
    cross PCIe instead of 12, and never on the critical path.  `host_images`: pinned tensors, one per view of this rank."""

    def __init__(self, host_images, device, slots=2):
        self.host = list(host_images)
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self.slots = [[torch.empty_like(h, device=self.device) for h in self.host] for _ in range(slots)]
        self.ready = [None] * slots
        self.consumed = [None] * slots
        self.head = 0                                  # next slot to fill
        self.tail = 0                                  # next slot to hand out
        self.bytes_per_step = sum(h.numel() * h.element_size() for h in self.host)

    def prefetch(self, host_images=None):
        src = self.host if host_images is None else host_images
        slot = self.head % len(self.slots)
        with torch.cuda.stream(self.stream):
            if self.consumed[slot] is not None:
                self.stream.wait_event(self.consumed[slot])      # the step that read this slot has finished with it
            for d, h in zip(self.slots[slot], src):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
            self.ready[slot] = ev
        self.head += 1

    def take(self):
        if self.tail == self.head:
            self.prefetch()
        slot = self.tail % len(self.slots)
        torch.cuda.current_stream().wait_event(self.ready[slot])
        self.tail += 1
        return self.slots[slot]

    def release(self):
        """Call after the step that used the last take() has been queued: its slot may be refilled once that work is done."""
        slot = (self.tail - 1) % len(self.slots)
        ev = torch.cuda.Event()
        ev.record()
        self.consumed[slot] = ev


class LossRing:
    """Per-step loss read-back without a host sync per step: the scalar is copied into a pinned ring asynchronously and read
    `lag` steps later (train_4DGS.py:236 calls loss.item() every iteration, which drains the GPU queue each time)."""

    def __init__(self, depth=4):
        self.host = torch.zeros(depth, dtype=torch.float32).pin_memory()
        self.events = [None] * depth
        self.n = 0

    def push(self, loss):
        i = self.n % self.host.numel()
        self.host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self.events[i] = ev
        self.n += 1

    def read(self, lag=1):
        """Value pushed `lag` steps ago (lag=0: the latest; waits for its copy only)."""
        if self.n - 1 - lag < 0:
            return None
        i = (self.n - 1 - lag) % self.host.numel()
        self.events[i].synchronize()
        return float(self.host[i])


def _receives_grad(name, stage):
    """Parameters the reference's loss reaches (SURVEY.md Appendix C iii): timenet, the opacity /
    SH heads and the aabb never do; in the coarse stage the whole deformation field is bypassed."""
    if name.startswith("_deformation."):
        if stage == "coarse":
            return False
        return not ("timenet" in name or "opacity_deform" in name or "shs_deform" in name or name.endswith("grid.aabb"))
    return True


class ViewParallelTrainer:
    """One optimiser step over a batch of views sharded across ranks (replicated model).

    `render_fn(cam, model, bg, stage)` defaults to this module's `render`; tests inject a CPU
    stand-in to exercise the sharding / flat-arena / collective logic over gloo.

    Step anatomy on the GPU (`shared_shs`, the default with our own render):
      * every trainable parameter except the two SH tensors has its `.grad` inside ONE flat FP32 arena
        `[xyz | MLP | planes | opacity | scaling | rotation | screen-space xy]`; the SH gradient -- 192 of the 260 bytes a
        Gaussian contributes -- lives in one `[P,16,3]` buffer that the rasterizer backward of every view adds into (the
        first view of a step overwrites it, so it is never zero-filled);
      * from inside the LAST view's backward -- right after its deformation-MLP backward has been queued (see step()) -- the SH
        tail starts on a side stream: `ncclAllReduce(sum)` of the SH buffer (+ the `max` of the radii), then the Adam step of
        the two SH tensors straight from that buffer (`FusedAdam.step_sh`) -- overlapping the time-plane / spatial HexPlane
        backward, the arena all-reduce and the plane regulariser on the main stream;
      * the main stream then reduces the (4x smaller) arena, adds the regulariser and takes the Adam step of everything
        else; the step ends by joining the side stream.
    Same sums, same Adam arithmetic as one collective + one optimiser launch (tests/test_dist_gloo.py, tests/test_dist_nccl.py)."""

    def __init__(self, model, bg_color, stage="fine", process_group=None, world_size=1, rank=0, render_fn=None,
                 regulation=None, regulation_fn=None, shared_shs=None, overlap_sh_reduce=None, lambda_dssim=0.0):
        self.model = model
        # opt.lambda_dssim (arguments/__init__.py): loss += lambda_dssim * (1 - ssim(image, gt)), fused path only; 0 = no D-SSIM term
        self.lambda_dssim = float(lambda_dssim)
        self.bg = bg_color
        self.stage = stage
        # (time_smoothness_weight, l1_time_planes, plane_tv_weight) of train_4DGS.py:215-218, or None to leave it out
        self.regulation = regulation if stage == "fine" else None
        self.regulation_fn = regulation_fn if stage == "fine" else None      # PyTorch-op variant (the reference arm of bench.py)
        self.pg = process_group
        self.world_size = world_size
        self.rank = rank
        # our own render() takes the per-step SH tensor; an injected render_fn keeps the 4-argument form
        self.shared_shs = (render_fn is None) if shared_shs is None else bool(shared_shs)
        self.render_fn = render_fn or (lambda cam, m, bg, st, shs=None, leaves=None: render(cam, m, bg, stage=st, shs=shs, leaves=leaves))
        self._own_render = render_fn is None
        dev = model.get_xyz.device
        # SH tail on a side stream, started from inside the last view's backward (B200GS_OVERLAP_SH_REDUCE=0: after the loop,
        # on the main stream -- same collectives, same order, nothing overlapped)
        if overlap_sh_reduce is None:
            overlap_sh_reduce = os.environ.get("B200GS_OVERLAP_SH_REDUCE", "1") != "0"
        self.overlap_sh_reduce = bool(overlap_sh_reduce) and self.shared_shs and dev.type == "cuda"
        self.side = torch.cuda.Stream(device=dev) if self.overlap_sh_reduce else None
        self._sh_started = False
        self._sh_done = None
        self._sse, self._sse_numel = None, 0
        # Forward of view i+1 on a second stream while view i's backward runs (B200GS_PIPELINE_VIEWS): the backwards stay
        # strictly ordered (every accumulator they share -- SH buffer, d(S), arena, viewspace, radii -- is touched in order),
        # only the latency-bound forward kernels (sorts, emission, read-back bubble) find idle SMs under the previous backward.
        self.pipeline_views = (os.environ.get("B200GS_PIPELINE_VIEWS", "1") != "0") and self.shared_shs and dev.type == "cuda"
        self.alt = torch.cuda.Stream(device=dev) if self.pipeline_views else None
        # streams the views rotate over (2: forward of view i+1 under the backward of view i; 3: view i+2's forward is queued too --
        # measured: 378 / 361-372 / 356 view-iters/s with 2 / 3 / 4 streams, so 2)
        self.pipeline_streams = max(2, int(os.environ.get("B200GS_PIPELINE_STREAMS", "2")))
        self.alts = ([self.alt] + [torch.cuda.Stream(device=dev) for _ in range(self.pipeline_streams - 2)]) if self.pipeline_views else []
        self.pipelined_mlp_sms = int(os.environ.get("B200GS_PIPELINED_MLP_SMS", "120"))      # 0: all SMs
        # SH tail from the rasterizer backward (instead of after the MLP backward) when the rank pipelines several views: the MLP
        # backward is confined to `pipelined_mlp_sms` SMs then, so the collective's CTAs no longer displace its persistent ones
        # (4 views per rank, N = 2: 661 -> 672 view-iters/s; 8 per rank, weak N = 4: 1,451 -> 1,496).  With one or two views per
        # rank the late start stays better (N = 8: 1,607 vs 1,575; N = 4: 1,102 vs 1,085): the confined MLP backward and the
        # collective's traffic slow the only views there are.  B200GS_SH_TAIL_EARLY=0/1 forces it.
        self.sh_tail_early = os.environ.get("B200GS_SH_TAIL_EARLY", "auto")
        self.timeline = None                           # bench.py: dict of CUDA events around the phases of the last step
        self._build_arena()

    def _build_arena(self):
        """(Re)creates the flat gradient arena for the model's CURRENT parameter tensors -- at construction and after every
        densification / pruning event (the per-Gaussian parameters are new, differently sized tensors then)."""
        model, stage = self.model, self.stage
        dev = model.get_xyz.device
        P = model.get_xyz.shape[0]
        # flat gradient arena: [every parameter the loss reaches except (shared_shs) the SH tensors | screen-space xy per
        # Gaussian]; p.grad are views into it, so autograd accumulates in place and ONE collective (fp32 sum over
        # NVLink/NVSwitch) reduces it. Parameters outside it keep grad None and the optimiser skips them, as torch does.
        named = [(n, p) for n, p in model.named_parameters() if p.requires_grad and _receives_grad(n, stage)]
        is_sh = lambda n: n in ("_features_dc", "_features_rest")
        self.sh_params = [p for n, p in named if is_sh(n)] if self.shared_shs else []
        if len(self.sh_params) != 2:
            self.sh_params = []
        arena_named = [x for x in named if not (self.sh_params and is_sh(x[0]))]
        self.trainable = [p for _, p in named]
        self.arena_params = [p for _, p in arena_named]
        # every slice starts on a 256-byte boundary: the kernels use 128-bit loads / vector reductions on them
        al = lambda x: (x + 63) // 64 * 64
        n = sum(al(p.numel()) for p in self.arena_params) + al(3 * P)
        self.arena = torch.zeros(n, dtype=torch.float32, device=dev)
        self.views, off = [], 0
        for name, p in arena_named:
            flat = self.arena[off:off + p.numel()]
            if p.dim() == 4 and p.stride(1) == 1 and not p.is_contiguous():     # channels_last plane
                N, C, H, W = p.shape
                v = flat.view(N, H, W, C).permute(0, 3, 1, 2)
            else:
                v = flat.view(p.shape)
            self.views.append(v)
            off += al(p.numel())
        self.viewspace_grad = self.arena[off:off + 3 * P].view(P, 3)
        self.max_radii = torch.zeros(P, dtype=torch.int32, device=dev)
        self.sh_grad = None                            # [P,M,3], allocated with the first step's SH tensor


    def rebuild(self):
        """Call after model.densify() / model.prune(): new arena, new SH gradient buffer."""
        self._build_arena()

    def _bind(self):
        self.arena.zero_()
        self.max_radii.zero_()
        for p, v in zip(self.arena_params, self.views):
            p.grad = v

    def _alias_leaves(self):
        """Second set of leaf tensors over the SAME storage and the SAME .grad buffers as the four per-Gaussian parameters the
        views reach through autograd (xyz, opacity, scaling, rotation), for the views rendered on the second stream.  A leaf's
        AccumulateGrad node runs on ONE stream -- the one its first forward use was recorded on -- so with a single set of
        leaves every odd view's backward (second stream) would hand its gradients to the first stream for accumulation, and the
        next view's forward, queued on that first stream, would wait for the end of that backward: no overlap for half of the
        views.  With its own leaves each stream accumulates by itself; the order of the adds is still the view order (the
        backwards are chained by events)."""
        m = self.model
        out = []
        for p in (m._xyz, m._opacity, m._scaling, m._rotation):
            a = p.detach().requires_grad_(p.requires_grad)
            a.grad = p.grad
            out.append(a)
        return tuple(out)

    def local_views(self, n_global):
        """Indices of the global batch this rank renders: view b goes to rank b mod world_size."""
        return list(range(self.rank, n_global, self.world_size))

    def _mark(self, name):
        if self.timeline is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.timeline[name] = ev

    # ---- SH tail: all-reduce of the SH gradient (+ radii max), then the SH parameters' Adam step ----------------------------
    def _sh_tail_body(self):
        import torch.distributed as dist
        m = self.model
        self._mark("sh_tail_start")
        if self.world_size > 1:
            dist.all_reduce(self.sh_grad, op=dist.ReduceOp.SUM, group=self.pg)
            dist.all_reduce(self.max_radii, op=dist.ReduceOp.MAX, group=self.pg)
        self._mark("sh_reduced")
        opt = m.optimizer
        if hasattr(opt, "step_sh") and self.sh_grad.is_cuda:
            opt.step_sh(m._features_dc, m._features_rest, self.sh_grad)
            self._sh_stepped = True
        else:                                          # any other optimiser: hand it the two slices, stepped with the rest
            m._features_dc.grad = self.sh_grad[:, :1]
            m._features_rest.grad = self.sh_grad[:, 1:]
            self._sh_stepped = False
        self._mark("sh_tail_end")

    def _sh_tail(self):
        """Called once per step: from the last view's rasterizer backward (overlap), else after the view loop."""
        if self._sh_started or not self.sh_params:
            return
        self._sh_started = True
        if self.side is None:
            self._sh_tail_body()
            return
        ready = torch.cuda.Event()
        ready.record()                                 # on the stream the rasterizer backward has just been queued on
        with torch.cuda.stream(self.side):
            self.side.wait_event(ready)
            self._sh_tail_body()
            self._sh_done = torch.cuda.Event()
            self._sh_done.record(self.side)

    def psnr(self):
        """utils/image_utils.py:psnr of the last step's LOCAL views, averaged (what train_4DGS.py:212 logs): a device tensor built
        from the squared-error sums the L1 kernel accumulated on the side; reading it is the caller's sync."""
        if self._sse is None:
            raise RuntimeError("psnr(): no step with views has run on this rank")
        return fusedops.psnr_from_sse(self._sse, self._sse_numel).mean()

    def step(self, cams, gts, global_batch=None):
        """cams / gts: THIS rank's views; a ground-truth image is a float32 [3,H,W] tensor or the dataset's own uint8 [H,W,3]
        image (GPU path). Loss = mean over the GLOBAL batch of per-view L1 means (train_4DGS.py:205-210: l1 over the
        concatenated [B,3,H,W] tensor), plus lambda_dssim * (1 - ssim) of the same batch when lambda_dssim > 0 (train_4DGS.py's
        opt.lambda_dssim term; the batch's SSIM is the mean of the per-view SSIMs since all views have the same size). Returns the
        summed local loss (already scaled by 1/B) as a tensor."""
        B = global_batch or (len(cams) * self.world_size)
        self._bind()
        self._mark("step_start")
        total = None
        sse_plain = []
        self._sse = None
        shs = None
        m = self.model
        self._sh_started, self._sh_done, self._sh_stepped = False, None, False
        if self.sh_params:
            # get_features (scene/gaussian_model.py:136-140) is the same tensor for every view of the step: build it once
            # as a leaf; every view's SH gradient accumulates in ONE buffer that outlives the step
            shs = torch.cat((m._features_dc, m._features_rest), dim=1).detach().requires_grad_(True)
            if self.sh_grad is None or self.sh_grad.shape != shs.shape:
                self.sh_grad = torch.zeros_like(shs)
            if shs.is_cuda:
                # the rasterizer backward adds every view's SH gradient straight into the buffer (the first view of the
                # step overwrites it): no per-view allocation, no zero fill, no AccumulateGrad pass over 192 B per Gaussian
                shs.grad = self.sh_grad
            m._features_dc.grad = None
            m._features_rest.grad = None
        from . import field as _field
        share_spatial = self.shared_shs and self.stage == "fine" and len(cams) > 1 and m._xyz.is_cuda
        if share_spatial:
            _field.begin_shared_step(m._deformation, m._xyz)
        first_sh = True
        import contextlib
        piped = self.pipeline_views and len(cams) > 1 and m._xyz.is_cuda
        main = torch.cuda.current_stream() if piped else None
        if piped:
            for st in self.alts:
                st.wait_stream(main)                   # shs, the spatial product and this step's images are ready
        ring = ([main] + self.alts) if piped else [None]
        stream_of = lambda vi: ring[vi % len(ring)]
        on = lambda st: torch.cuda.stream(st) if st is not None else contextlib.nullcontext()

        alias = [None] + [self._alias_leaves() for _ in self.alts] if piped and self._own_render else None
        depth = len(ring) - 1 if piped else 1          # forwards queued ahead of the backward in progress
        early = (piped and self.world_size > 1 and len(cams) >= 4) if self.sh_tail_early == "auto" else (self.sh_tail_early != "0" and self.world_size > 1)
        confine = (piped or early) and self.pipelined_mlp_sms
        if confine:
            # the deformation-MLP kernels are persistent, one CTA per SM with 157 / 230 KB of shared memory: while they own every SM
            # nothing of the other stream's forward can be resident.  Leaving them 120 of the 148 SMs costs them little (they are
            # latency-bound) and lets the sorts / emission / preprocess of the next view run next to them (377 -> 383 view-iters/s).
            from . import _lib
            for name in (b"mlp_bwd_sms", b"mlp_fwd_sms"):
                _lib.lib().b200gs_set_option(name, int(self.pipelined_mlp_sms))

        def forward_view(vi):
            with on(stream_of(vi)):
                if alias is not None and alias[vi % len(ring)] is not None:
                    return self.render_fn(cams[vi], m, self.bg, self.stage, shs, alias[vi % len(ring)])
                return self.render_fn(cams[vi], m, self.bg, self.stage, shs) if self.shared_shs else \
                    self.render_fn(cams[vi], m, self.bg, self.stage)
        prev_done = None
        try:
            ahead = [forward_view(k) for k in range(min(depth, len(cams)))]
            for vi, (cam, gt) in enumerate(zip(cams, gts)):
                pkg = ahead.pop(0)
                with on(stream_of(vi)):
                    if prev_done is not None:
                        torch.cuda.current_stream().wait_event(prev_done)
                    # (before the backward: the SH tail, which reduces max_radii over the ranks, starts from inside the LAST one)
                    torch.maximum(self.max_radii, pkg["radii"], out=self.max_radii)
                    _field.ACCUMULATE_INTO_GRAD = self.shared_shs     # p.grad are arena views: let the field kernels add into them
                    on_gpu = shs is not None and shs.is_cuda
                    _rast.SH_GRAD_ACCUMULATOR = self.sh_grad if on_gpu else None
                    _rast.SH_GRAD_OVERWRITE = first_sh
                    if on_gpu and self.overlap_sh_reduce and vi == len(cams) - 1:
                        # The SH tail starts from inside the LAST view's backward.  The SH gradient is complete as soon as the
                        # rasterizer backward has been queued, but the deformation-MLP backward that follows is a persistent kernel
                        # with one 230 KB CTA per SM and a static tile schedule: a collective that holds a few SMs while it runs
                        # delays those CTAs by the collective's whole duration (measured at N = 8: 0.60 -> 1.22 ms).  So the tail
                        # is started right AFTER the MLP backward has been queued and overlaps the time-plane / spatial HexPlane
                        # backward, the arena all-reduce and the regulariser instead -- ordinary kernels that share SMs gracefully.
                        if self.stage == "fine" and hasattr(_field, "AFTER_MLP_BACKWARD") and not early:
                            _field.AFTER_MLP_BACKWARD = self._sh_tail
                        else:
                            _rast.AFTER_SH_ACCUMULATE = self._sh_tail
                    try:
                        if self.shared_shs and gt.is_cuda:
                            # fused L1 (utils/loss_utils.py:23-24) + its gradient, then backward from the image
                            if total is None:          # [loss | one squared-error sum per local view] zeroed by one fill
                                acc_buf = torch.zeros(1 + len(cams), device=gt.device)
                                total, self._sse = acc_buf[:1], acc_buf[1:]
                            img = pkg["render"]
                            self._sse_numel = img.numel()
                            d_img = fusedops.l1_loss_and_grad(img, gt, 1.0 / (img.numel() * B), total, self._sse[vi:])
                            if self.lambda_dssim > 0.0:
                                # + lambda_dssim * (1 - ssim) of this view's share, its gradient added into d_img
                                fusedops.dssim_loss_and_grad(img, gt, self.lambda_dssim / B, total, d_img)
                            img.backward(d_img)
                            loss = None
                        else:
                            if self.lambda_dssim > 0.0:
                                raise NotImplementedError("lambda_dssim > 0 needs the fused path (our own render on the GPU)")
                            diff = pkg["render"] - gt
                            loss = diff.abs().mean() / B
                            sse_plain.append((diff.detach() ** 2).sum().reshape(1))
                            self._sse_numel = diff.numel()
                            loss.backward()
                    finally:
                        _field.ACCUMULATE_INTO_GRAD = False
                        _rast.SH_GRAD_ACCUMULATOR = None
                        _rast.SH_GRAD_OVERWRITE = False
                        _rast.AFTER_SH_ACCUMULATE = None
                        _field.AFTER_MLP_BACKWARD = None
                    first_sh = False
                    vg = pkg["viewspace_points"].grad
                    if vg is not None:
                        self.viewspace_grad += vg
                    if loss is not None:
                        total = loss.detach() if total is None else total + loss.detach()
                    if piped:
                        prev_done = torch.cuda.Event()
                        prev_done.record()
                del pkg
                if vi + depth < len(cams):
                    # piped: on ANOTHER stream, so it runs under the backward queued just above (its stage-1 read-back is
                    # the only host wait of a view, and that backward keeps the GPU busy meanwhile)
                    ahead.append(forward_view(vi + depth))
            if piped and prev_done is not None:
                main.wait_event(prev_done)
        except BaseException:
            _field.drop_shared()               # never leave a half-used spatial product behind (a later render() would reuse it)
            raise
        finally:
            if confine:
                from . import _lib
                for name in (b"mlp_bwd_sms", b"mlp_fwd_sms"):
                    _lib.lib().b200gs_set_option(name, 0)
        if sse_plain:
            self._sse = torch.cat(sse_plain)
        self._mark("views_done")
        if self.sh_params:
            if not shs.is_cuda:                        # CPU plumbing tests: autograd accumulated into the leaf itself
                self.sh_grad = shs.grad if shs.grad is not None else torch.zeros_like(shs)
            elif first_sh:                             # a rank without views still takes part in the collective
                self.sh_grad.zero_()
            self._sh_tail()                            # no-op when the last view's backward has already started it
        if share_spatial:
            _field.finish_shared_step()
        self._mark("field_done")
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(self.arena, op=dist.ReduceOp.SUM, group=self.pg)
            if not self.sh_params:
                dist.all_reduce(self.max_radii, op=dist.ReduceOp.MAX, group=self.pg)
        self._mark("arena_reduced")
        if self.regulation is not None:
            # plane-only term, identical on every rank: added once, after the reduce (SURVEY.md 8e)
            # (its VALUE goes into rank 0's share of the loss only, so that the shares still sum to the global loss)
            fused_total = total is not None and total.numel() == 1 and total.dim() == 1
            acc = total if fused_total else (torch.zeros(1, device=self.arena.device) if total is not None else None)
            _field.accumulate_regulation(m._deformation.deformation_net.grid, *self.regulation,
                                         loss_accum=acc if self.rank == 0 else None)
            if not fused_total and acc is not None and self.rank == 0:
                total = total + acc.reshape(())
        if self.regulation_fn is not None:
            reg = self.regulation_fn()
            reg.backward()
            total = total + reg.detach()
        if self._sh_done is not None:
            # join BEFORE the main-stream optimiser launch when the SH tensors were not stepped on the side stream
            if not self._sh_stepped:
                torch.cuda.current_stream().wait_event(self._sh_done)
        if self._sh_stepped:
            m.optimizer.step(skip=tuple(self.sh_params))
        else:
            m.optimizer.step()
        self._mark("adam_done")
        if self._sh_done is not None and self._sh_stepped:
            torch.cuda.current_stream().wait_event(self._sh_done)
        self._mark("step_end")
        return total.reshape(()) if total is not None else total
