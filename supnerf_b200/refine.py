"""Refine-iteration glue around the render hot path (SURVEY.md §8f rank 1): the test-time optimisation loop of
``optimizer_nuscenes.py:684-769`` (identical in optimizer_kitti.py / optimizer_waymo.py) for ONE object --

    rot_vec, trans_vec -> cam2opt                         (:684-699; the axis-angle map is pytorch3d's, one step upstream of the path)
    render_rays_v2(model, ..., cam2opt, ...)              (:716-726 -> utils.py:435-502)
    loss_rgb + loss_occ_coef * loss_occ ; backward        (:729-737)
    AdamW step on shapecode, texturecode, rot_vec, trans_vec   (:757-769, groups/lrs of :1762-1769)

-- with every host synchronisation removed so that one iteration can be captured in a CUDA graph and replayed: the
reference reads ``cam_pose[:, -1].tolist()`` on the host every iteration to build the shared sample vector
(utils.py:468-469 -> sample_from_rays :154-167); here near/far are evaluated on the device with the same arithmetic
(float64 norm, float32 ``torch.linspace`` formula), and the per-iteration jitter -- drawn on the CPU generator by the
same ``torch.rand(n_samples)`` calls, in the same order -- is uploaded once as a table.  ``ms per refine iteration``
then is kernel time (~25 launches replayed from one graph: 0.21 ms at 32x32 rays on a B200) instead of ~2.4 ms of
Python / launch latency.

The render, loss and their backward are the package's fused kernels (ops.render_shell, losses.refine_loss); with
``fused=True`` (default) the pose map + sample vectors and the AdamW update are single launches too (csrc/refine.cu:
snb_refine_pose_slots_fwd / snb_refine_pose_batch_bwd, snb_adamw_step_rows -- the same launches BatchRefiner and SlotRefiner issue
for many objects, here with one row); ``fused=False`` keeps them as torch ops (torch.optim.AdamW(capturable=True)) -- the tests
check both against the loop written with the reference-shaped API.  CUDA only."""
import ctypes
import math

import numpy as np
import torch

from . import _lib, losses, models, ops
from . import utils as U
from ._lib import check, f32c, on_device, ptr, require_cuda, stream_ptr


class SlotAdamW:
    """torch.optim.AdamW's update on `rows` independent rows of a handful of small tensors (one row per object or refine slot) in ONE
    launch (snb_adamw_step_rows); state lives on the device.  Each row has its own step counter (``step_t`` (rows,)), which also picks
    its jitter row in the pose map, and active byte (``active`` (rows,) uint8); an inactive row is left bit-for-bit unchanged."""

    def __init__(self, groups, rows, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2):
        self.params = [g["params"] for g in groups]
        self.lrs = [float(g["lr"]) for g in groups]
        self.betas, self.eps, self.weight_decay = betas, eps, weight_decay
        dev = self.params[0].device
        self.rows = int(rows)
        self.m = [torch.zeros_like(p) for p in self.params]
        self.v = [torch.zeros_like(p) for p in self.params]
        self.step_t = torch.zeros(self.rows, device=dev, dtype=torch.float32)
        self.active = torch.ones(self.rows, device=dev, dtype=torch.uint8)
        n = len(self.params)
        self._sizes = (ctypes.c_int32 * n)(*[p.numel() // self.rows for p in self.params])
        self._lrs = (ctypes.c_float * n)(*self.lrs)

    def zero_grad(self, set_to_none=True):
        """set_to_none (default): the next backward ASSIGNS the gradients instead of accumulating into zero-filled ones: no fill
        and no add kernel per parameter (inside a CUDA graph the assigned tensors keep their addresses across replays)."""
        for p in self.params:
            if p.grad is not None:
                if set_to_none:
                    p.grad = None
                else:
                    p.grad.zero_()

    def reset_row(self, r):
        """Zero row r's moments and step counter (stream-ordered, no host synchronisation)."""
        for t in self.m + self.v:
            t[r].zero_()
        self.step_t[r].zero_()

    def step(self, loss3=None, loss_rgb2=None, history=None):
        """One update of every active row.  history (rows, T, 4) (optional): an active row r first writes [loss3[r, 0:3], loss_rgb2[r]] to
        history[r, step_t[r]] (loss3 (rows,3) contiguous, loss_rgb2 a (rows,) view with any row stride)."""
        lib = _lib.load()
        n = len(self.params)
        arr = lambda ts: (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])  # noqa: E731
        stride = int(loss_rgb2.stride(0)) if loss_rgb2 is not None else 0
        t_rows = int(history.shape[1]) if history is not None else 0
        with on_device(self.params[0].device):
            check(lib.snb_adamw_step_rows(n, arr(self.params), arr([p.grad for p in self.params]), arr(self.m), arr(self.v), self._sizes, self._lrs,
                                          self.betas[0], self.betas[1], self.eps, self.weight_decay, self.rows, ptr(self.step_t), ptr(self.active),
                                          ptr(loss3), ptr(loss_rgb2), stride, ptr(history), t_rows, stream_ptr()), "snb_adamw_step_rows")


class _PoseAndSamplesBatch(torch.autograd.Function):
    """(B,3) rot_vec, trans_vec -> cam2opt (B,3,4) + every object's shared sample vector z (B,S) [+ a second one, z2, from another jitter
    table] in ONE launch (snb_refine_pose_slots_fwd).  Object b reads row step_t[b] of its jitter tables (B, T, S) -- its optimiser's step
    counter; an active object (`active` (B,) uint8) whose counter lies outside the table gets NaN samples and sets `err` (optional)."""

    @staticmethod
    def forward(ctx, rot_vec, trans_vec, jitter, jitter2, step_t, obj_diag, opt_cam_pose, n_samples, active, err=None):
        lib = _lib.load()
        require_cuda(rot_vec, trans_vec, jitter, step_t, obj_diag, active)
        rot_vec, trans_vec = f32c(rot_vec), f32c(trans_vec)
        b, t, s = jitter.shape
        dev = rot_vec.device
        cam = torch.empty(b, 3, 4, device=dev, dtype=torch.float32)
        z = torch.empty(b, s, device=dev, dtype=torch.float32)
        z2 = torch.empty(b, s, device=dev, dtype=torch.float32) if jitter2 is not None else None
        with on_device(dev):
            check(lib.snb_refine_pose_slots_fwd(ptr(rot_vec), ptr(trans_vec), int(b), int(bool(opt_cam_pose)), ptr(obj_diag), int(n_samples),
                                                ptr(jitter), ptr(jitter2), ptr(step_t), int(t), ptr(active), ptr(err), ptr(cam), ptr(z),
                                                ptr(z2), stream_ptr()), "snb_refine_pose_slots_fwd")
        ctx.save_for_backward(rot_vec, trans_vec)
        ctx.opt_cam_pose = int(bool(opt_cam_pose))
        ctx.set_materialize_grads(False)
        if z2 is None:
            ctx.mark_non_differentiable(z)
            return cam, z
        ctx.mark_non_differentiable(z, z2)
        return cam, z, z2

    @staticmethod
    def backward(ctx, g_cam, *_):
        lib = _lib.load()
        rot_vec, trans_vec = ctx.saved_tensors
        if g_cam is None:
            return (None,) * 10
        g_cam = f32c(g_cam)
        g_rot, g_trans = torch.empty_like(rot_vec), torch.empty_like(trans_vec)
        with on_device(rot_vec.device):
            check(lib.snb_refine_pose_batch_bwd(ptr(rot_vec), ptr(trans_vec), int(rot_vec.shape[0]), ctx.opt_cam_pose, ptr(g_cam), ptr(g_rot),
                                                ptr(g_trans), stream_ptr()), "snb_refine_pose_batch_bwd")
        return (g_rot, g_trans) + (None,) * 8


def _capture(device, warm_up, body):
    """Run warm_up() on a side stream (allocator, weight packing, AdamW state), then record body() into a CUDA graph.  The capture
    itself does not execute: the state after it is the one warm_up() left."""
    s = torch.cuda.Stream(device=device)
    s.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(s):
        warm_up()
    torch.cuda.current_stream(device).wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    return graph


def _reserve(refiners, iters):
    """Count `iters` more iterations of every ObjectRefiner against its pre-drawn jitter tables, before any of them is issued.
    -> iters.  ValueError, counting nothing, if one of them would read past its tables."""
    iters = int(iters)
    if iters < 0 or any(iters > r.remaining for r in refiners):
        raise ValueError("iters exceeds the pre-drawn jitter table (max_iters)")
    for r in refiners:
        r.remaining -= iters
    return iters


def axis_angle_to_matrix(v):
    """Rodrigues' formula, R = I + sin(t)/t [v]x + (1-cos(t))/t^2 [v]x^2 -- what pytorch3d.transforms.axis_angle_to_matrix
    evaluates (via quaternions); pytorch3d itself is not part of the reference tree (SURVEY §8c: parity unpinned there)."""
    t = torch.sqrt((v * v).sum() + 1e-20)
    zero = torch.zeros((), device=v.device, dtype=v.dtype)
    kx = torch.stack([torch.stack([zero, -v[2], v[1]]), torch.stack([v[2], zero, -v[0]]), torch.stack([-v[1], v[0], zero])])
    return torch.eye(3, device=v.device, dtype=v.dtype) + torch.sin(t) / t * kx + (1 - torch.cos(t)) / (t * t) * (kx @ kx)


def shell_samples_on_device(cam_pose, obj_diag, n_samples, jitter):
    """utils.sample_from_rays' shared vector (utils.py:154-167 with near/far of :468-469) without leaving the device.
    near/far: float64 like the reference's python floats; linspace: torch's float32 formula (step = (end-start)/(n-1);
    first half start + i*step, second half end - (n-1-i)*step); jitter (S,) = the torch.rand(n_samples) draw."""
    n = torch.linalg.vector_norm(cam_pose[:, -1].detach().double())
    half = float(obj_diag) / 2          # obj_diag is np.float32 in the reference: exactly representable
    near, far = n - half, n + half
    dist = (far - near) / (2 * n_samples)
    start, end = (near + dist).float(), (far - dist).float()
    step = (end - start) / (n_samples - 1) if n_samples > 1 else torch.zeros_like(start)
    i = torch.arange(n_samples, device=cam_pose.device, dtype=torch.float32)
    lo = start + step * i
    hi = end - step * (n_samples - 1 - i)
    z = torch.where(i < n_samples // 2, lo, hi)
    return z + jitter * ((far - near) / (2 * n_samples)).float()


class ObjectRefiner:
    """One object's refine loop.  ``step()`` runs one iteration eagerly; ``capture()`` records it into a CUDA graph and
    ``run(n)`` replays it.  State (codes, pose parameters, AdamW moments) lives in this object's tensors."""

    def __init__(self, model, device, img, mask_occ, K, roi, obj_diag, shapecode, texturecode, rot_vec, trans_vec, n_samples=64,
                 im_sz=32, lr_shape=0.02, lr_texture=0.02, lr_pose=0.01, loss_occ_coef=0.1, shapenet_obj_cood=True,
                 opt_cam_pose=False, max_iters=100, fused=True, lidar_xy=None):
        if not isinstance(model, models._DecoderBase):
            raise TypeError("ObjectRefiner needs a supnerf_b200 decoder")
        self.model, self.device = model, torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("supnerf_b200 has no CPU path")
        dev = self.device
        self.n_samples, self.im_sz, self.coef = int(n_samples), int(im_sz), float(loss_occ_coef)
        self.obj_diag, self.swap, self.opt_cam_pose = np.float32(obj_diag), bool(shapenet_obj_cood), bool(opt_cam_pose)
        self.K = K.to(dev, torch.float32)
        self.px, self.py = U._pixel_grid_on(dev, roi, [im_sz, im_sz])
        img, mask_occ = U._resize_targets(img, mask_occ, im_sz)          # utils.py:448-453
        self.rgb_tgt = img.reshape(-1, 3).to(dev).contiguous()
        self.occ = mask_occ.reshape(-1, 1).to(dev).contiguous()
        self.shapecode = shapecode.detach().to(dev).clone().requires_grad_()
        self.texturecode = texturecode.detach().to(dev).clone().requires_grad_()
        self.rot_vec = rot_vec.detach().to(dev).reshape(3).clone().requires_grad_()
        self.trans_vec = trans_vec.detach().to(dev).reshape(3).clone().requires_grad_()
        # fused = True: pose map + sample vectors and the AdamW update as single launches (csrc/refine.cu, one row); False: torch ops
        self.fused = bool(fused)
        if self.fused:
            self.opt = SlotAdamW([{"params": self.shapecode, "lr": lr_shape}, {"params": self.texturecode, "lr": lr_texture},
                                  {"params": self.rot_vec, "lr": lr_pose}, {"params": self.trans_vec, "lr": lr_pose}], rows=1)
        else:
            self.opt = torch.optim.AdamW([{"params": [self.shapecode], "lr": lr_shape}, {"params": [self.texturecode], "lr": lr_texture},
                                          {"params": [self.rot_vec], "lr": lr_pose}, {"params": [self.trans_vec], "lr": lr_pose}],
                                         capturable=True)
        # Per-iteration evaluation the reference interleaves with the optimisation (optimizer_nuscenes.py:740-769): the PSNR loss over
        # the object mask only (loss_rgb2) and a no-grad depth render of the pixels that carry a lidar return (render_rays_specified).
        # lidar_xy = (x_vec, y_vec): integer pixel offsets inside the crop (np.where of the depth map, :759); None = not evaluated.
        self.lidar, self.n_lidar = None, 0
        if lidar_xy is not None:
            x_vec, y_vec = np.asarray(lidar_xy[0]), np.asarray(lidar_xy[1])
            self.n_lidar = int(x_vec.shape[0])
            if self.n_lidar > 0:
                lx = torch.from_numpy(x_vec + int(roi[0])).reshape(-1).to(dev, torch.float32)
                ly = torch.from_numpy(y_vec + int(roi[1])).reshape(-1).to(dev, torch.float32)
                pad = (-self.n_lidar) % 2            # the bf16 decoder works on 128-row tiles: an even ray count at 64 samples
                if pad:
                    lx, ly = torch.cat([lx, lx[-1:]]), torch.cat([ly, ly[-1:]])
                self.lidar = (lx.contiguous(), ly.contiguous())
        self.occ_pos = self.occ.clamp_min(0.0)       # mask_rgb: occ_pixels with the negative (background) entries zeroed (:741-742)
        self.loss_rgb2 = torch.zeros((), device=dev)
        self.depth_pred = torch.zeros(0, device=dev)
        # the reference draws torch.rand(n_samples) on the CPU generator once per render call (utils.py:164): per iteration one draw
        # for the optimised render and, when the lidar pixels are evaluated, a second one for render_rays_specified -- same calls, same order
        per_it = 2 if self.lidar is not None else 1
        draws = torch.stack([torch.rand(self.n_samples) for _ in range(max_iters * per_it)]).to(dev)
        self.jitter = draws[0::per_it].contiguous()
        self.jitter_lidar = draws[1::per_it].contiguous() if self.lidar is not None else None
        self.remaining = int(max_iters)   # host-side count of the iterations left in the jitter tables (eager steps and replays alike)
        if self.fused:                     # the jitter row is the optimiser's step counter
            self.obj_diag_dev = torch.tensor([float(self.obj_diag)], device=dev)
        else:                              # the jitter row of the next iteration
            self.it = torch.zeros((), dtype=torch.long, device=dev)
        self.loss = torch.zeros(3, device=dev)
        self.graph = None

    def cam2opt(self):
        rot = axis_angle_to_matrix(self.rot_vec)
        t = self.trans_vec.unsqueeze(-1)
        if not self.opt_cam_pose:                     # optimizer_nuscenes.py:695-697
            rot = rot.transpose(-2, -1)
            t = -rot @ t
        return torch.cat((rot, t), dim=-1)

    def step(self):
        """One iteration, eagerly (no host synchronisation anywhere)."""
        _reserve([self], 1)
        return self._iteration()

    def _iteration(self):
        if self.shapecode.grad is not None:
            self.opt.zero_grad() if self.fused else self.opt.zero_grad(set_to_none=False)
        if self.fused:   # (1, 3) views of the pose parameters, (1, T, S) views of the jitter tables
            out = _PoseAndSamplesBatch.apply(self.rot_vec.view(1, 3), self.trans_vec.view(1, 3), self.jitter[None],
                                             None if self.lidar is None else self.jitter_lidar[None], self.opt.step_t, self.obj_diag_dev,
                                             self.opt_cam_pose, self.n_samples, self.opt.active)
            cam, z = out[0].view(3, 4), out[1].view(-1)
        else:
            jit = self.jitter.index_select(0, self.it.reshape(1)).reshape(-1)
            cam = self.cam2opt()
            z = shell_samples_on_device(cam, self.obj_diag, self.n_samples, jit)
        prec = self.model.precision or models.get_default_precision()
        rgb, dep, acc = ops.render_shell(self.model._handle(self.device), prec, self.n_samples, float(self.obj_diag), self.swap,
                                         self.px, self.py, self.K, cam, z, self.shapecode, self.texturecode, self.model._weights())
        loss, vec = losses.refine_loss_vec(rgb, acc, self.rgb_tgt, self.occ, self.coef)
        loss.backward()
        with torch.no_grad():       # the per-iteration evaluation (optimizer_nuscenes.py:740-769), before the parameter update as there
            self.loss_rgb2 = losses.refine_loss(rgb.detach(), acc.detach(), self.rgb_tgt, self.occ_pos, 0.0)[1]
            if self.lidar is not None:
                if self.fused:
                    z2 = out[2].view(-1)
                else:
                    jit2 = self.jitter_lidar.index_select(0, self.it.reshape(1)).reshape(-1)
                    z2 = shell_samples_on_device(cam.detach(), self.obj_diag, self.n_samples, jit2)
                _, dep2, _ = ops.render_shell(self.model._handle(self.device), prec, self.n_samples, float(self.obj_diag), self.swap,
                                              self.lidar[0], self.lidar[1], self.K, cam.detach(), z2, self.shapecode.detach(),
                                              self.texturecode.detach(), self.model._weights())
                self.depth_pred = dep2[:self.n_lidar]
        self.opt.step()
        self.loss = vec   # [loss, loss_rgb, loss_occ] as the loss kernel wrote them (graph mode: a static tensor of the graph's pool)
        if not self.fused:
            self.it += 1
        return self.loss

    def _warm_up(self, steps):
        """`steps` iterations on the current stream that leave the refine state as it was.  Fused: with the active byte cleared, so
        nothing is updated or counted and the jitter row stays inside the table; else: undone from a snapshot, each from row 0."""
        if self.fused:
            self.opt.active.zero_()
            for _ in range(steps):
                self._iteration()
            self.opt.active.fill_(1)
            return
        state = (self.shapecode, self.texturecode, self.rot_vec, self.trans_vec, self.it)
        snapshot = [t.detach().clone() for t in state]
        for _ in range(steps):
            self.it.zero_()
            self._iteration()
        with torch.no_grad():       # parameters, iteration counter, AdamW moments and step counters
            for t, v in zip(state, snapshot):
                t.copy_(v)
            for st in self.opt.state.values():
                for v in st.values():
                    if torch.is_tensor(v):
                        v.zero_()

    def capture(self, warmup=3):
        """Warm up on a side stream, then capture one iteration."""
        self.graph = _capture(self.device, lambda: self._warm_up(warmup), self._iteration)
        return self

    def run(self, iters):
        """Run `iters` iterations (graph replays if captured).  Returns the last [loss, loss_rgb, loss_occ] (device tensor).
        ValueError, issuing nothing, if they would run past the pre-drawn jitter table (max_iters iterations in all)."""
        for _ in range(_reserve([self], iters)):
            if self.graph is not None:
                self.graph.replay()
            else:
                self._iteration()
        return self.loss


def run_objects(refiners, iters, n_streams=4):
    """Refine several INDEPENDENT objects side by side (SURVEY 8e, object-parallel: own pose, codes, rays, loss and AdamW state):
    iteration k of every object is issued round-robin over `n_streams` CUDA streams, so one object's small kernels (pose map,
    sampler, compositing, loss, AdamW) run under another object's decoder kernel instead of leaving the GPU idle between two
    decoder launches.  No host synchronisation; the caller's current stream waits for all of them at the end.
    Returns the objects' last [loss, loss_rgb, loss_occ] tensors."""
    if not refiners:
        return []
    dev = refiners[0].device
    main = torch.cuda.current_stream(dev)
    streams = [torch.cuda.Stream(device=dev) for _ in range(max(1, min(int(n_streams), len(refiners))))]
    for s in streams:
        s.wait_stream(main)
    for _ in range(int(iters)):
        for i, r in enumerate(refiners):
            with torch.cuda.stream(streams[i % len(streams)]):
                r.run(1)
    for s in streams:
        main.wait_stream(s)
    return [r.loss for r in refiners]


class ObjectGroup:
    """Several INDEPENDENT objects (config C3: a GPU's 4 of the 32 objects) refined side by side from ONE CUDA graph per iteration:
    the capture forks the objects' iterations onto one stream each and joins them, so a replay is a single graph launch whose
    branches the device schedules concurrently (one object's ~30 small kernels under another's decoder kernel) -- instead of one
    graph launch per object per iteration issued round-robin from the host (run_objects)."""

    def __init__(self, refiners):
        if not refiners:
            raise ValueError("ObjectGroup needs at least one refiner")
        self.refiners = list(refiners)
        self.device = self.refiners[0].device
        self.graph = None

    def capture(self, warmup=3):
        """Warm up every object on a side stream (ObjectRefiner's warm-up), then capture one iteration of all of them."""
        dev = self.device
        streams = [torch.cuda.Stream(device=dev) for _ in self.refiners]

        def iteration():
            main = torch.cuda.current_stream(dev)
            for s_, r in zip(streams, self.refiners):
                s_.wait_stream(main)                 # fork
                with torch.cuda.stream(s_):
                    r._iteration()
            for s_ in streams:
                main.wait_stream(s_)                 # join

        def warm_up():
            for r in self.refiners:
                r._warm_up(warmup)
        self.graph = _capture(dev, warm_up, iteration)
        return self

    def run(self, iters):
        """`iters` iterations of every object.  -> the objects' last [loss, loss_rgb, loss_occ] tensors.  ValueError, issuing nothing, if
        one object would run past its pre-drawn jitter table."""
        for _ in range(_reserve(self.refiners, iters)):
            if self.graph is not None:
                self.graph.replay()
            else:
                for r in self.refiners:
                    r._iteration()
        return [r.loss for r in self.refiners]


class SlotRefiner:
    """A stream of INDEPENDENT objects refined through C fixed slots (the reference's test-time refinement goes through the evaluation split
    one object at a time: optimize_objs_w_pose_unified, optimizer_nuscenes.py:684-769).  Each slot holds one object's refine state; one
    iteration of all C slots is ONE launch set (ObjectRefiner's iteration over every slot at once), captured ONCE as a CUDA graph.
    Between replays the host ``admit``s an ObjectRefiner into a free slot with its own iteration budget, and ``run`` retires every object
    whose budget is used up, copying its results back into its ObjectRefiner -- all stream-ordered, without a host synchronisation.  The
    host knows every slot's remaining budget without reading the device: each replay advances every active slot by exactly one iteration.

    Every slot has its own AdamW step counter (SlotAdamW), which also picks its jitter row, and an active byte.  A free slot keeps running
    on finite placeholder inputs (a fixed synthetic object at first, its last object's inputs with zero loss weights after a retirement):
    it takes no AdamW step, writes no loss history and reports nothing, but its render is paid.  ``max_lidar`` is the per-slot capacity of
    lidar pixels evaluated every iteration (0 = no lidar evaluation).  ``capture()`` may come before or after admissions."""

    def __init__(self, model, device, slots=16, n_samples=64, im_sz=32, max_iters=100, max_lidar=0, lr_shape=0.02, lr_texture=0.02,
                 lr_pose=0.01, loss_occ_coef=0.1, shapenet_obj_cood=True, opt_cam_pose=False):
        if not isinstance(model, models._DecoderBase):
            raise TypeError("SlotRefiner needs a supnerf_b200 decoder")
        self.model, self.device = model, torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("supnerf_b200 has no CPU path")
        if int(slots) < 1 or int(max_iters) < 1 or int(max_lidar) < 0:
            raise ValueError("SlotRefiner: slots >= 1, max_iters >= 1, max_lidar >= 0")
        dev = self.device
        c, s, n = int(slots), int(n_samples), int(im_sz) ** 2
        self.slots, self.n_samples, self.im_sz, self.max_iters = c, s, int(im_sz), int(max_iters)
        self.coef, self.swap, self.opt_cam_pose = float(loss_occ_coef), bool(shapenet_obj_cood), bool(opt_cam_pose)
        d = model._latent_dim
        # placeholder object (finite everywhere, zero loss weights): camera 2.5 units from the origin looking down +z, unit diagonal
        px, py = U._pixel_grid_on(dev, [0, 0, int(im_sz), int(im_sz)], [int(im_sz), int(im_sz)])
        self.px = px.reshape(1, -1).repeat(c, 1).contiguous()
        self.py = py.reshape(1, -1).repeat(c, 1).contiguous()
        f = float(im_sz)
        self.K = torch.tensor([[f, 0.0, f / 2], [0.0, f, f / 2], [0.0, 0.0, 1.0]], device=dev).repeat(c, 1, 1).contiguous()
        self.rgb_tgt = torch.zeros(c, n, 3, device=dev)
        self.occ = torch.zeros(c, n, device=dev)
        self.occ_pos = torch.zeros(c, n, device=dev)
        self.obj_diag = torch.ones(c, device=dev)
        self.shapecode = torch.zeros(c, d, device=dev).requires_grad_()
        self.texturecode = torch.zeros(c, d, device=dev).requires_grad_()
        self.rot_vec = torch.zeros(c, 3, device=dev).requires_grad_()
        self.trans_vec = torch.tensor([0.0, 0.0, 2.5], device=dev).repeat(c, 1).contiguous().requires_grad_()
        self.opt = SlotAdamW([{"params": self.shapecode, "lr": lr_shape}, {"params": self.texturecode, "lr": lr_texture},
                              {"params": self.rot_vec, "lr": lr_pose}, {"params": self.trans_vec, "lr": lr_pose}], rows=c)
        self.opt.active.zero_()
        self.jitter = torch.zeros(c, self.max_iters, s, device=dev)
        self.lidar, self.jitter_lidar, self.width = None, None, 0
        if int(max_lidar) > 0:   # whole 256-row decoder super tiles per slot: 4 rays at 64 samples
            q = 256 // math.gcd(256, s)
            self.width = -(-int(max_lidar) // q) * q
            self.lidar = (self.px[:, :1].repeat(1, self.width).contiguous(), self.py[:, :1].repeat(1, self.width).contiguous())
            self.jitter_lidar = torch.zeros(c, self.max_iters, s, device=dev)
        self.history = torch.zeros(c, self.max_iters, 4, device=dev)   # [loss, loss_rgb, loss_occ, loss_rgb2] per slot and iteration
        self.err = torch.zeros(1, device=dev, dtype=torch.int32)       # set by the pose kernel if an active slot's counter leaves its table
        self._ones = torch.ones(c, device=dev)
        self.loss = torch.zeros(c, 3, device=dev)
        self.loss_rgb2 = torch.zeros(c, device=dev)
        self.depth_pred = None
        self.owner = [None] * c          # the ObjectRefiner in each slot (None = free)
        self.budget = [0] * c            # its iteration budget
        self.remaining = [0] * c         # iterations it still has to run
        self.n_lidar = [0] * c
        self.replays = 0                 # host-side counts: slot-iterations issued, and those of occupied slots
        self.busy_slot_iters = 0
        self.graph = None

    def _iteration(self):
        """ObjectRefiner's iteration for every slot at once (no host synchronisation anywhere)."""
        if self.shapecode.grad is not None:
            self.opt.zero_grad()
        out = _PoseAndSamplesBatch.apply(self.rot_vec, self.trans_vec, self.jitter, self.jitter_lidar, self.opt.step_t, self.obj_diag,
                                         self.opt_cam_pose, self.n_samples, self.opt.active, self.err)
        cam, z = out[0], out[1]
        prec = self.model.precision or models.get_default_precision()
        h, w = self.model._handle(self.device), self.model._weights()
        rgb, _dep, acc = ops.render_shell_batch(h, prec, self.n_samples, self.swap, self.px, self.py, self.K, cam, z, self.obj_diag,
                                                self.shapecode, self.texturecode, w)
        loss, parts = losses.refine_loss_batch(rgb, acc, self.rgb_tgt, self.occ, self.coef)
        torch.autograd.backward(loss, self._ones)
        with torch.no_grad():       # the per-iteration evaluation (optimizer_nuscenes.py:740-769), before the parameter update as there
            self.loss_rgb2 = losses.refine_loss_batch(rgb.detach(), acc.detach(), self.rgb_tgt, self.occ_pos, 0.0)[1][:, 1]
            if self.lidar is not None:
                _, dep2, _ = ops.render_shell_batch(h, prec, self.n_samples, self.swap, self.lidar[0], self.lidar[1], self.K, cam.detach(),
                                                    out[2], self.obj_diag, self.shapecode.detach(), self.texturecode.detach(), w)
                self.depth_pred = dep2           # (C, width): slot b's lidar depths are depth_pred[b, :n_lidar[b]]
        self.loss = parts           # (C,3) = [loss, loss_rgb, loss_occ] per slot
        self.opt.step(self.loss, self.loss_rgb2, self.history)
        return self.loss

    def _warm_up(self, steps):
        """`steps` iterations with every active byte cleared: nothing is updated or counted and every slot reads a row inside its jitter
        tables, so nothing needs restoring."""
        active = self.opt.active.clone()
        self.opt.active.zero_()
        for _ in range(steps):
            self._iteration()
        self.opt.active.copy_(active)

    def capture(self, warmup=3):
        """Warm up on a side stream (allocator, weight packing), then capture one iteration of all slots, occupied or free."""
        self.graph = _capture(self.device, lambda: self._warm_up(warmup), self._iteration)
        return self

    def free_slots(self):
        return [b for b, o in enumerate(self.owner) if o is None]

    def busy(self):
        return any(o is not None for o in self.owner)

    def admit(self, r, iters):
        """Put ObjectRefiner `r` into a free slot with a budget of `iters` iterations (stream-ordered copies, no host synchronisation).
        -> the slot index.  ValueError if its settings differ from this refiner's, there is no free slot, `iters` exceeds max_iters or the
        object's jitter rows, or it has more lidar pixels than the slot capacity."""
        iters = int(iters)
        lrs = (float(self.opt.lrs[0]), float(self.opt.lrs[1]), float(self.opt.lrs[2]), float(self.opt.lrs[2]))
        if not (r.model is self.model and r.device == self.device and r.fused and (r.n_samples, r.im_sz, r.coef, r.swap, r.opt_cam_pose)
                == (self.n_samples, self.im_sz, self.coef, self.swap, self.opt_cam_pose) and tuple(r.opt.lrs) == lrs
                and (tuple(r.opt.betas), r.opt.eps, r.opt.weight_decay) == (tuple(self.opt.betas), self.opt.eps, self.opt.weight_decay)):
            raise ValueError("SlotRefiner.admit: the object must share the decoder, device, n_samples, crop size, loss and optimiser settings "
                             "(and be a fused ObjectRefiner)")
        if not 1 <= iters <= min(self.max_iters, r.jitter.shape[0]):
            raise ValueError("SlotRefiner.admit: iters must be in 1 .. min(max_iters, the object's jitter rows)")
        n_lidar = r.n_lidar
        if n_lidar > self.width:
            raise ValueError("SlotRefiner.admit: %d lidar pixels exceed the slot capacity (%d)" % (n_lidar, self.width))
        free = self.free_slots()
        if not free:
            raise ValueError("SlotRefiner.admit: no free slot")
        b = free[0]
        k = min(self.max_iters, r.jitter.shape[0])
        with torch.no_grad():
            self.px[b].copy_(r.px.reshape(-1))
            self.py[b].copy_(r.py.reshape(-1))
            self.K[b].copy_(r.K)
            self.rgb_tgt[b].copy_(r.rgb_tgt)
            self.occ[b].copy_(r.occ.reshape(-1))
            self.occ_pos[b].copy_(r.occ_pos.reshape(-1))
            self.obj_diag[b].fill_(float(r.obj_diag))
            self.shapecode[b].copy_(r.shapecode.detach().reshape(-1))
            self.texturecode[b].copy_(r.texturecode.detach().reshape(-1))
            self.rot_vec[b].copy_(r.rot_vec.detach())
            self.trans_vec[b].copy_(r.trans_vec.detach())
            self.jitter[b, :k].copy_(r.jitter[:k])
            if self.lidar is not None:
                if n_lidar:
                    x, y = r.lidar[0][:n_lidar], r.lidar[1][:n_lidar]
                    self.jitter_lidar[b, :k].copy_(r.jitter_lidar[:k])
                else:   # no lidar pixels: a dummy pixel is rendered and nothing reported
                    x, y = r.px.reshape(-1)[:1], r.py.reshape(-1)[:1]
                    self.jitter_lidar[b].zero_()
                self.lidar[0][b, :x.numel()].copy_(x)
                self.lidar[0][b, x.numel():].copy_(x[-1:].expand(self.width - x.numel()))
                self.lidar[1][b, :y.numel()].copy_(y)
                self.lidar[1][b, y.numel():].copy_(y[-1:].expand(self.width - y.numel()))
            self.opt.reset_row(b)
            self.history[b].zero_()
            self.opt.active[b].fill_(1)
        self.owner[b], self.budget[b], self.remaining[b], self.n_lidar[b] = r, iters, iters, n_lidar
        return b

    def _copy_out(self, b):
        """Copy slot b's results into its ObjectRefiner: codes, pose parameters, last losses, lidar depths and loss_history (iterations
        run, 4)."""
        r, n = self.owner[b], self.n_lidar[b]
        with torch.no_grad():
            r.shapecode.copy_(self.shapecode[b].reshape(r.shapecode.shape))
            r.texturecode.copy_(self.texturecode[b].reshape(r.texturecode.shape))
            r.rot_vec.copy_(self.rot_vec[b])
            r.trans_vec.copy_(self.trans_vec[b])
            r.loss = self.loss[b].clone()          # copies: the slot's buffers are rewritten by the next replay
            r.loss_rgb2 = self.loss_rgb2[b].clone()
            if n and self.depth_pred is not None:
                r.depth_pred = self.depth_pred[b, :n].clone()
            r.loss_history = self.history[b, :self.budget[b] - self.remaining[b]].clone()

    def _retire(self, b):
        """Copy slot b's results into its ObjectRefiner and free the slot."""
        self._copy_out(b)
        with torch.no_grad():
            self.opt.active[b].fill_(0)
            # zero loss weights: the idle slot's upstream gradients are exactly zero, so the batched backward skips its decoder tiles
            self.occ[b].zero_()
            self.occ_pos[b].zero_()
        self.owner[b], self.remaining[b] = None, 0

    def step(self):
        """One iteration of every slot, eagerly; counted and retired as a replay is."""
        return self._advance(1, eager=True)

    def run(self, iters):
        """`iters` iterations of every slot (graph replays if captured); an object whose budget is used up is retired right after its last
        iteration.  -> (C,3) last [loss, loss_rgb, loss_occ] per slot (device tensor)."""
        return self._advance(int(iters))

    def _advance(self, iters, eager=False):
        """Issue `iters` iterations (graph replays unless eager or not captured) and count them on the host, slot by slot."""
        for _ in range(iters):
            if self.graph is None or eager:
                self._iteration()
            else:
                self.graph.replay()
            self.replays += 1
            for b in range(self.slots):
                if self.owner[b] is not None:
                    self.busy_slot_iters += 1
                    self.remaining[b] -= 1
                    if self.remaining[b] == 0:
                        self._retire(b)
        return self.loss

    def stream(self, refiners, iters):
        """Refine every ObjectRefiner of `refiners` (iters: one budget for all, or one per object), admitting the next one as soon as a slot
        is free, so every slot stays busy while objects remain.  Ends with a synchronisation (raises if the kernels' error flag is set).
        Returns the refiners in input order, their results written back (codes, pose parameters, last losses, lidar depths, loss_history)."""
        refiners = list(refiners)
        budgets = [int(i) for i in iters] if hasattr(iters, "__len__") else [int(iters)] * len(refiners)
        if len(budgets) != len(refiners):
            raise ValueError("SlotRefiner.stream: one budget per refiner")
        todo = list(zip(refiners, budgets))[::-1]
        while todo or self.busy():
            for _ in self.free_slots():
                if todo:
                    self.admit(*todo.pop())
            self.run(min(self.remaining[b] for b in range(self.slots) if self.owner[b] is not None))
        self.synchronize()
        return refiners

    def idle_share(self):
        """Share of the slot-iterations issued so far that ran on a free slot."""
        total = self.replays * self.slots
        return 1.0 - self.busy_slot_iters / total if total else 0.0

    def synchronize(self):
        """Wait for the device, then raise if an active slot read outside its jitter table (the kernels' error flag)."""
        torch.cuda.current_stream(self.device).synchronize()
        if int(self.err.item()):
            raise RuntimeError("SlotRefiner: an active slot's step counter left its jitter table (its sample vectors are NaN)")


def refine_stream(refiners, iters, slots=16):
    """Refine ObjectRefiners through one SlotRefiner of min(slots, len(refiners)) slots with their settings (SlotRefiner.stream).
    iters: one budget for all, or one per object.  Returns the refiners in input order, results written back."""
    refiners = list(refiners)
    if not refiners:
        return []
    budgets = [int(i) for i in iters] if hasattr(iters, "__len__") else [int(iters)] * len(refiners)
    sr = SlotRefiner(refiners[0].model, refiners[0].device, slots=min(int(slots), len(refiners)), max_iters=max(budgets),
                     max_lidar=max(r.n_lidar for r in refiners), **_settings(refiners[0]))
    return sr.capture().stream(refiners, budgets)


def _settings(r):
    """SlotRefiner's sample count, crop size, learning rates, loss coefficient and axis conventions from ObjectRefiner r's."""
    lrs = r.opt.lrs
    return dict(n_samples=r.n_samples, im_sz=r.im_sz, lr_shape=lrs[0], lr_texture=lrs[1], lr_pose=lrs[2], loss_occ_coef=r.coef,
                shapenet_obj_cood=r.swap, opt_cam_pose=r.opt_cam_pose)


class BatchRefiner(SlotRefiner):
    """The refine loops of B INDEPENDENT objects (one GPU's share of config C3) as ONE launch set per iteration: every stage of
    ObjectRefiner.step -- pose map + sample vectors, the utils.py-stack render, the losses, their backward, the per-iteration
    evaluation (loss_rgb2, lidar-pixel depths) and the AdamW update -- runs once over all objects (ops.render_shell_batch,
    losses.refine_loss_batch, snb_refine_pose_slots_fwd / snb_refine_pose_batch_bwd, snb_adamw_step_rows), ~25 launches per iteration
    whatever B is instead of ~30 per object.  The objects stay independent: per-object pose, codes, rays, targets, jitter draws, losses
    (the summed loss has block-diagonal gradients) and elementwise AdamW state.

    A SlotRefiner with one slot per object, every slot admitted for the objects' whole jitter tables and never retired.  Built from
    ObjectRefiners (which hold the per-object inputs and the jitter tables drawn in the reference's order); they must agree on n_samples,
    crop size, learning rates, loss coefficient, axis convention, decoder and jitter rows.  ``write_back()`` copies the optimised state
    into them."""

    def __init__(self, refiners):
        if not refiners:
            raise ValueError("BatchRefiner needs at least one refiner")
        r0 = refiners[0]
        same = lambda f: all(f(r) == f(r0) for r in refiners)   # noqa: E731
        if not (same(lambda r: (r.n_samples, r.im_sz, r.coef, r.swap, r.opt_cam_pose, r.fused, tuple(r.opt.lrs) if r.fused else None,
                                r.jitter.shape[0])) and all(r.model is r0.model and r.device == r0.device for r in refiners)):
            raise ValueError("BatchRefiner: the objects must share the decoder, device, n_samples, crop size, loss and optimiser settings")
        if not r0.fused:
            raise ValueError("BatchRefiner builds on the fused refiners (fused=True)")
        super().__init__(r0.model, r0.device, slots=len(refiners), max_iters=r0.jitter.shape[0], max_lidar=max(r.n_lidar for r in refiners),
                         **_settings(r0))
        self.refiners = list(refiners)
        for r in self.refiners:
            self.admit(r, self.max_iters)

    def step(self):
        """One iteration of every object, eagerly.  ValueError if the jitter tables are used up."""
        self._check(1)
        return self._advance(1, eager=True)

    def run(self, iters):
        """`iters` iterations of every object (graph replays if captured).  -> (B,3) last [loss, loss_rgb, loss_occ] per object.
        ValueError, issuing nothing, if they would run past the pre-drawn jitter tables (max_iters iterations in all)."""
        self._check(iters)
        return self._advance(int(iters))

    def _check(self, iters):
        if int(iters) < 0 or int(iters) > min(self.remaining):
            raise ValueError("iters exceeds the pre-drawn jitter tables (max_iters)")

    def _retire(self, b):
        """Objects stay in their slots when their tables are used up: write_back() copies their state out."""

    def lidar_depths(self):
        """Per object: the depths at its lidar pixels from the last iteration's evaluation (None for an object without lidar pixels)."""
        if self.depth_pred is None:
            return [None] * len(self.refiners)
        return [self.depth_pred[b, :n] if n else None for b, n in enumerate(self.n_lidar)]

    def write_back(self):
        """Copy the optimised codes, pose parameters and last results into the ObjectRefiners this batch was built from; the objects
        stay in their slots."""
        for b in range(self.slots):
            self._copy_out(b)
        return self.refiners
