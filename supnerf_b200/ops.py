"""torch.autograd bindings of the C-ABI kernels.  Each Function cites the reference code it replaces.

All tensors handed to the library are CUDA fp32 contiguous; outputs are fresh tensors attached to the
autograd graph.  No function here has a CPU or eager-PyTorch fallback."""
import ctypes
import os

import numpy as np
import torch

from . import _lib
from ._lib import check, f32c, on_device, ptr, require_cuda, stream_ptr

WHITE_BKGD, SIGMA_RELU = 1, 2
PREC = {"fp32": 0, "bf16": 1}
PREC_BF16_TRAIN = 2  # selected automatically in bf16 mode when a weight requires grad (SNB_PREC_BF16_TRAIN)
PREC_FP32_TC = 3     # selected automatically in fp32 mode when NO weight takes a gradient (SNB_PREC_FP32_TC): the same 1e-5 parity
#                      on the tensor cores (two fp16 parts per operand, three MMAs per product), ~20x the FFMA back end's throughput
FP32_TENSOR_CORES = os.environ.get("SNB_FP32_SIMT", "0") in ("", "0")   # False: fp32 mode always runs the FFMA kernels


FP32_TC_MAX_WEIGHT = 255.0   # 256 * w must stay inside fp16's range (csrc/mlp_tc.cu: kWScale)


def _fp32_tc(handle, prec, rows_per_obj=None, weights=None):
    """fp32 mode with frozen weights -> the split-precision tensor-core kernels where they apply (CodeNeRF family, W = 128 or 256;
    dense row counts a multiple of the 128-row tile; every |weight| < 255 -- checked once per weight version).  rows_per_obj None: the
    caller's rows are compacted on the device (any count)."""
    if prec != PREC["fp32"] or not FP32_TENSOR_CORES or not handle.tc_ok:
        return prec
    if rows_per_obj is not None and (rows_per_obj <= 0 or rows_per_obj % 128 != 0):
        return prec
    if weights is not None and not handle.weights_in_fp16_range(weights):
        return prec
    return PREC_FP32_TC


# ---------------------------------------------------------------------------------------------------
# K3 / K3b  — renderer.py:43-65, :355-379; utils.py:187-233
# ---------------------------------------------------------------------------------------------------
class _Composite(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sigma, rgb, z, rays_per_zrow, flags):
        lib = _lib.load()
        require_cuda(sigma, rgb, z)
        sigma, rgb, z = f32c(sigma), f32c(rgb), f32c(z)
        n, s = sigma.shape
        o_rgb = torch.empty(n, 3, device=sigma.device, dtype=torch.float32)
        o_dep = torch.empty(n, device=sigma.device, dtype=torch.float32)
        o_acc = torch.empty(n, device=sigma.device, dtype=torch.float32)
        with on_device(sigma.device):
            check(lib.snb_composite_fwd(ptr(sigma), ptr(rgb), ptr(z), rays_per_zrow, n, s, flags, ptr(o_rgb), ptr(o_dep),
                                        ptr(o_acc), stream_ptr()), "snb_composite_fwd")
        ctx.save_for_backward(sigma, rgb, z)
        ctx.meta = (rays_per_zrow, flags)
        return o_rgb, o_dep, o_acc

    @staticmethod
    def backward(ctx, g_rgb, g_dep, g_acc):
        lib = _lib.load()
        sigma, rgb, z = ctx.saved_tensors
        rays_per_zrow, flags = ctx.meta
        n, s = sigma.shape
        g_rgb = f32c(g_rgb) if g_rgb is not None else torch.zeros(n, 3, device=sigma.device)
        g_dep = f32c(g_dep) if g_dep is not None else torch.zeros(n, device=sigma.device)
        g_acc = f32c(g_acc) if g_acc is not None else torch.zeros(n, device=sigma.device)
        g_sigma = torch.empty_like(sigma)
        g_rgbs = torch.empty_like(rgb)
        need_z = ctx.needs_input_grad[2]
        g_z = torch.empty_like(sigma) if need_z else None
        with on_device(sigma.device):
            check(lib.snb_composite_bwd(ptr(sigma), ptr(rgb), ptr(z), rays_per_zrow, n, s, flags, ptr(g_rgb), ptr(g_dep),
                                        ptr(g_acc), ptr(g_sigma), ptr(g_rgbs), ptr(g_z), stream_ptr()), "snb_composite_bwd")
        if need_z and z.shape[0] != n:  # shared rows: reduce the per-ray gradient onto the shared vector(s)
            g_z = g_z.reshape(z.shape[0], rays_per_zrow, s).sum(1)
        return g_sigma, g_rgbs, g_z, None, None


def composite(sigma, rgb, z, white_bkgd, relu=True):
    """sigma (N,S), rgb (N,S,3); z (N,S) per ray, (S,) shared, or (B,S) with N = B*n."""
    n, s = sigma.shape
    if z.dim() == 1:
        zz, rpz = z.reshape(1, s), max(n, 1)
    else:
        zz, rpz = z, max(n // max(z.shape[0], 1), 1)
    flags = (WHITE_BKGD if white_bkgd else 0) | (SIGMA_RELU if relu else 0)
    rgb_o, dep, acc = _Composite.apply(sigma, rgb, zz, rpz, flags)
    return rgb_o, dep, acc


# ---------------------------------------------------------------------------------------------------
# K1 / K1b — utils.py:107-151 (rays), :283-327 (slab), renderer.py:91-115 (box sampler), utils.py:154-167
# ---------------------------------------------------------------------------------------------------
class _GetRays(torch.autograd.Function):
    @staticmethod
    def forward(ctx, px, py, K, c2w):
        lib = _lib.load()
        require_cuda(px, py, K, c2w)
        px, py, K, c2w = f32c(px), f32c(py), f32c(K), f32c(c2w)
        n = px.numel()
        ro = torch.empty(n, 3, device=px.device, dtype=torch.float32)
        vd = torch.empty(n, 3, device=px.device, dtype=torch.float32)
        with on_device(px.device):
            check(lib.snb_get_rays_fwd(ptr(px), ptr(py), n, ptr(K), ptr(c2w), ptr(ro), ptr(vd), stream_ptr()), "snb_get_rays_fwd")
        ctx.save_for_backward(px, py, K, c2w)
        return ro, vd

    @staticmethod
    def backward(ctx, g_ro, g_vd):
        lib = _lib.load()
        px, py, K, c2w = ctx.saved_tensors
        n = px.numel()
        g_ro = f32c(g_ro) if g_ro is not None else torch.zeros(n, 3, device=px.device)
        g_vd = f32c(g_vd) if g_vd is not None else torch.zeros(n, 3, device=px.device)
        g_c2w = torch.zeros(3, 4, device=px.device, dtype=torch.float32)
        with on_device(px.device):
            check(lib.snb_get_rays_bwd(ptr(px), ptr(py), n, ptr(K), ptr(c2w), ptr(g_ro), ptr(g_vd), ptr(g_c2w), stream_ptr()),
                  "snb_get_rays_bwd")
        return None, None, None, g_c2w


def get_rays_from_pixels(px, py, K, c2w):
    return _GetRays.apply(px, py, K, c2w)


class _RayBox(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ro, rd, amin, amax):
        lib = _lib.load()
        require_cuda(ro, rd, amin, amax)
        ro, rd = f32c(ro), f32c(rd)
        amin = f32c(amin) if amin is not None else None
        amax = f32c(amax) if amax is not None else None
        n = ro.shape[0]
        tn = torch.empty(n, device=ro.device, dtype=torch.float32)
        tf = torch.empty(n, device=ro.device, dtype=torch.float32)
        hit = torch.empty(n, device=ro.device, dtype=torch.uint8)
        with on_device(ro.device):
            check(lib.snb_ray_box_fwd(ptr(ro), ptr(rd), ptr(amin), ptr(amax), n, ptr(tn), ptr(tf), ptr(hit), stream_ptr()),
                  "snb_ray_box_fwd")
        ctx.save_for_backward(ro, rd, amin, amax)
        hitb = hit.bool()
        ctx.mark_non_differentiable(hitb)
        return tn, tf, hitb

    @staticmethod
    def backward(ctx, g_tn, g_tf, _g_hit):
        lib = _lib.load()
        ro, rd, amin, amax = ctx.saved_tensors
        n = ro.shape[0]
        g_tn = f32c(g_tn) if g_tn is not None else torch.zeros(n, device=ro.device)
        g_tf = f32c(g_tf) if g_tf is not None else torch.zeros(n, device=ro.device)
        g_o, g_d = torch.empty_like(ro), torch.empty_like(rd)
        g_min = torch.empty_like(ro) if amin is not None and ctx.needs_input_grad[2] else None
        g_max = torch.empty_like(ro) if amax is not None and ctx.needs_input_grad[3] else None
        with on_device(ro.device):
            check(lib.snb_ray_box_bwd(ptr(ro), ptr(rd), ptr(amin), ptr(amax), n, ptr(g_tn), ptr(g_tf), ptr(g_o), ptr(g_d),
                                      ptr(g_min), ptr(g_max), stream_ptr()), "snb_ray_box_bwd")
        return g_o, g_d, g_min, g_max


def ray_box(ro, rd, amin=None, amax=None):
    """Uncompacted (t_near, t_far, hit)."""
    return _RayBox.apply(ro, rd, amin, amax)


class _SampleBox(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rays_o, viewdir, z_steps, jitter, half_diag, aabb_half, detach_bounds=False):
        lib = _lib.load()
        require_cuda(rays_o, viewdir, z_steps, jitter)
        rays_o, viewdir, z_steps, jitter = f32c(rays_o), f32c(viewdir), f32c(z_steps), f32c(jitter)
        n, s = jitter.shape
        dev = rays_o.device
        xyz = torch.empty(n, s, 3, device=dev, dtype=torch.float32)
        vrep = torch.empty(n, s, 3, device=dev, dtype=torch.float32)
        zv = torch.empty(n, s, device=dev, dtype=torch.float32)
        hit = torch.empty(n, device=dev, dtype=torch.uint8)
        h3 = (ctypes.c_float * 3)(*[float(v) for v in aabb_half])
        with on_device(dev):
            check(lib.snb_sample_box_fwd(ptr(rays_o), ptr(viewdir), ptr(z_steps), ptr(jitter), n, s, float(half_diag), h3,
                                         ptr(xyz), ptr(vrep), ptr(zv), ptr(hit), stream_ptr()), "snb_sample_box_fwd")
        ctx.save_for_backward(rays_o, viewdir, z_steps, jitter)
        ctx.meta = (float(half_diag), [float(v) for v in aabb_half], int(bool(detach_bounds)))
        hitb = hit.bool()
        ctx.mark_non_differentiable(hitb)
        return xyz, vrep, zv, hitb

    @staticmethod
    def backward(ctx, g_xyz, g_vrep, g_zv, _g_hit):
        lib = _lib.load()
        rays_o, viewdir, z_steps, jitter = ctx.saved_tensors
        half_diag, half, detach = ctx.meta
        n, s = jitter.shape
        g_xyz = f32c(g_xyz) if g_xyz is not None else None
        g_vrep = f32c(g_vrep) if g_vrep is not None else None
        g_zv = f32c(g_zv) if g_zv is not None else None
        g_o, g_d = torch.empty_like(rays_o), torch.empty_like(viewdir)
        h3 = (ctypes.c_float * 3)(*half)
        with on_device(rays_o.device):
            check(lib.snb_sample_box_bwd(ptr(rays_o), ptr(viewdir), ptr(z_steps), ptr(jitter), n, s, half_diag, h3, ptr(g_xyz),
                                         ptr(g_vrep), ptr(g_zv), ptr(g_o), ptr(g_d), detach, stream_ptr()), "snb_sample_box_bwd")
        return g_o, g_d, None, None, None, None, None


def jitter_fill(seed, n_rays, n_samples, device, ray_ids=None):
    """(n_rays, S) stratified jitter in [0, 1) as a pure function of (seed, ray id, sample index) (snb_jitter_fill: Philox4x32-10):
    a rank of the ray-sharded mode fills only ITS rows (`ray_ids`: int64 ids of its rays) and the union over the ranks equals the
    one-GPU fill bit for bit.  Not the reference's torch.rand_like stream."""
    lib = _lib.load()
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("supnerf_b200 has no CPU path")
    if ray_ids is not None:
        require_cuda(ray_ids)
        ray_ids = ray_ids.to(torch.int64).contiguous()
        n_rays = ray_ids.numel()
    out = torch.empty(int(n_rays), int(n_samples), device=device, dtype=torch.float32)
    with on_device(device):
        check(lib.snb_jitter_fill(int(seed) & 0xFFFFFFFFFFFFFFFF, ptr(ray_ids), int(n_rays), int(n_samples), ptr(out), stream_ptr()), "snb_jitter_fill")
    return out


def sample_box(rays_o, viewdir, z_steps, jitter, half_diag, aabb_half, detach_bounds=False):
    """renderer.py:91-115 in one kernel.  detach_bounds: the slab test's near / far carry no gradient (renderer.render_rays_v3 runs it
    on detached host copies of the rays, renderer.py:425-432)."""
    return _SampleBox.apply(rays_o, viewdir, z_steps, jitter, half_diag, aabb_half, detach_bounds)


class _StratifiedZ(torch.autograd.Function):
    """renderer.py:27-41 = utils.py:170-184 on its own: rays (N, C) with near / far in the last two columns -> z (N, S)."""

    @staticmethod
    def forward(ctx, rays, z_steps, jitter):
        lib = _lib.load()
        require_cuda(rays, z_steps, jitter)
        rays, z_steps, jitter = f32c(rays), f32c(z_steps), f32c(jitter)
        n, s = jitter.shape
        z = torch.empty(n, s, device=rays.device, dtype=torch.float32)
        with on_device(rays.device):
            check(lib.snb_stratified_z_fwd(ptr(rays), int(rays.shape[1]), ptr(z_steps), ptr(jitter), n, s, ptr(z), stream_ptr()),
                  "snb_stratified_z_fwd")
        ctx.save_for_backward(z_steps, jitter)
        ctx.cols = int(rays.shape[1])
        return z

    @staticmethod
    def backward(ctx, g_z):
        lib = _lib.load()
        z_steps, jitter = ctx.saved_tensors
        n, s = jitter.shape
        g_z = f32c(g_z)
        g_rays = torch.zeros(n, ctx.cols, device=jitter.device, dtype=torch.float32)
        g_near = torch.empty(n, device=jitter.device, dtype=torch.float32)
        g_far = torch.empty(n, device=jitter.device, dtype=torch.float32)
        with on_device(jitter.device):
            check(lib.snb_stratified_z_bwd(ptr(z_steps), ptr(jitter), n, s, ptr(g_z), ptr(g_near), ptr(g_far), stream_ptr()),
                  "snb_stratified_z_bwd")
        g_rays[:, -2] = g_near
        g_rays[:, -1] = g_far
        return g_rays, None, None


def stratified_z(rays, z_steps, jitter):
    return _StratifiedZ.apply(rays, z_steps, jitter)


class _SampleShell(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rays_o, viewdir, z, obj_diag, swap):
        lib = _lib.load()
        require_cuda(rays_o, viewdir, z)
        rays_o, viewdir, z = f32c(rays_o), f32c(viewdir), f32c(z)
        n, s = rays_o.shape[0], z.numel()
        xyz = torch.empty(n, s, 3, device=rays_o.device, dtype=torch.float32)
        vrep = torch.empty(n, s, 3, device=rays_o.device, dtype=torch.float32)
        with on_device(rays_o.device):
            check(lib.snb_sample_shell_fwd(ptr(rays_o), ptr(viewdir), ptr(z), n, s, float(obj_diag), int(swap), ptr(xyz),
                                           ptr(vrep), stream_ptr()), "snb_sample_shell_fwd")
        ctx.save_for_backward(z)
        ctx.meta = (n, s, float(obj_diag), int(swap))
        return xyz, vrep

    @staticmethod
    def backward(ctx, g_xyz, g_vrep):
        lib = _lib.load()
        (z,) = ctx.saved_tensors
        n, s, obj_diag, swap = ctx.meta
        g_xyz = f32c(g_xyz) if g_xyz is not None else None
        g_vrep = f32c(g_vrep) if g_vrep is not None else None
        g_o = torch.empty(n, 3, device=z.device, dtype=torch.float32)
        g_d = torch.empty(n, 3, device=z.device, dtype=torch.float32)
        with on_device(z.device):
            check(lib.snb_sample_shell_bwd(ptr(z), n, s, obj_diag, swap, ptr(g_xyz), ptr(g_vrep), ptr(g_o), ptr(g_d),
                                           stream_ptr()), "snb_sample_shell_bwd")
        return g_o, g_d, None, None, None


def sample_shell(rays_o, viewdir, z, obj_diag=1.0, shapenet_swap=False):
    return _SampleShell.apply(rays_o, viewdir, z, obj_diag, shapenet_swap)


# ---------------------------------------------------------------------------------------------------
# K2 / K2b — model_codenerf.py:39-63 ≡ model_autorf.py:226-250 ≡ model_supnerf.py:241-269; model_autorf.py:156-186
# ---------------------------------------------------------------------------------------------------
class DecoderHandle:
    """One C handle per (module, device): borrowed fp32 weight pointers + (bf16 mode) the packed images."""

    def __init__(self, arch, shape_blocks, texture_blocks, W, latent_dim, num_xyz_freq, num_dir_freq):
        lib = _lib.load()
        self.arch = _lib.SnbArch(arch, shape_blocks, texture_blocks, W, latent_dim, num_xyz_freq, num_dir_freq)
        self.h = ctypes.c_void_p()
        check(lib.snb_create(ctypes.byref(self.h), ctypes.byref(self.arch)), "snb_create")
        self.n_tensors = lib.snb_num_weight_tensors(self.h)
        self._packed = None
        self._packed_key = None
        self._keep = None
        self._frozen = None
        self.tc_ok = lib.snb_packed_bytes(self.h) > 16      # the tensor-core back ends cover this architecture

    def __del__(self):
        try:
            if self.h:
                _lib.load().snb_destroy(self.h)
        except Exception:
            pass

    def set_weights(self, tensors, saved=False):
        """Point the handle at the fp32 weight storages.  saved=True (an autograd backward re-presenting the tensors its forward
        saved): the forward already set exactly these storages unless another forward ran in between, so comparing the first
        and last pointer is enough to skip the full key."""
        lib = _lib.load()
        assert len(tensors) == self.n_tensors, (len(tensors), self.n_tensors)
        old = self.__dict__.get("_set_key")
        if saved and old is not None and tensors[0].data_ptr() == old[0] and tensors[-1].data_ptr() == old[-1]:
            return
        key = tuple([t.data_ptr() for t in tensors])
        if key == old and all([t.dtype == torch.float32 and t.is_contiguous() for t in tensors]):
            return   # same storage as last time: the handle already borrows these pointers
        self._set_key = key
        self._keep = [f32c(t.detach()) for t in tensors]
        require_cuda(*self._keep)
        arr = (ctypes.c_void_p * self.n_tensors)(*[t.data_ptr() for t in self._keep])
        check(lib.snb_set_weights(self.h, arr, self.n_tensors), "snb_set_weights")

    def use_frozen(self, tensors, precision):
        """Point the handle at a weight set that takes no part in autograd; `_frozen` identifies the set last used."""
        self.set_weights(tensors)
        if precision != PREC["fp32"]:
            self.ensure_packed(tensors)
        if self.__dict__.get("_frozen") is not tensors:
            self._frozen = tensors

    def weights_in_fp16_range(self, tensors):
        """True when every weight is finite and below FP32_TC_MAX_WEIGHT in magnitude (the split-precision kernels hold 256 * w in
        fp16 pairs).  One device reduction + read-back per weight version; the answer is cached with the version key."""
        key = self.packed_key(tensors)
        hit = self.__dict__.get("_range_key")
        if hit is not None and hit[0] == key:
            return hit[1]
        if torch.cuda.is_current_stream_capturing():
            return True      # no read-back inside a capture: the warm-up iterations before it have answered for these weights
        with torch.no_grad():
            biggest = float(torch.stack([t.detach().abs().max() for t in tensors if t.numel()]).max())
        ok = biggest == biggest and biggest < FP32_TC_MAX_WEIGHT
        self._range_key = (key, ok)
        return ok

    def invalidate_packed(self):
        """Force a re-pack of the bf16 weight images at the next call.  Needed after weight edits autograd's version counter does
        not see (``p.data.copy_(...)``, ``p.data.mul_(...)``: EMA updates, manual checkpoint loading idioms); ordinary in-place
        updates (optimisers, ``p.copy_`` under no_grad) bump the counter and are picked up automatically."""
        self._packed_key = None

    def packed_key(self, tensors):
        return tuple((t.data_ptr(), t._version) for t in tensors)

    def ensure_packed(self, tensors):
        """bf16 mode: (re)pack when a parameter was replaced or modified in place."""
        lib = _lib.load()
        key = self.packed_key(tensors)
        if key == self._packed_key and self._packed is not None:
            return
        nbytes = lib.snb_packed_bytes(self.h)
        dev = self._keep[0].device
        if self._packed is None or self._packed.numel() < nbytes or self._packed.device != dev:
            self._packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with on_device(dev):
            check(lib.snb_pack_weights(self.h, ptr(self._packed), stream_ptr()), "snb_pack_weights")
        self._packed_key = key


class _Decoder(torch.autograd.Function):
    @staticmethod
    def forward(ctx, handle, precision, n_objs, xyz, viewdir, shape_latent, texture_latent, *weights):
        lib = _lib.load()
        require_cuda(xyz, viewdir, shape_latent, texture_latent)
        xyz, viewdir = f32c(xyz), f32c(viewdir)
        shape_latent, texture_latent = f32c(shape_latent), f32c(texture_latent)
        m = xyz.numel() // 3
        dev = xyz.device
        handle.set_weights(weights)
        if precision == PREC["fp32"] and not any(ctx.needs_input_grad[7:]):
            precision = _fp32_tc(handle, precision, m // max(n_objs, 1), weights)
        if precision == PREC["bf16"]:
            handle.ensure_packed(weights)
            if any(ctx.needs_input_grad[7:]):
                precision = PREC_BF16_TRAIN   # keep the operand tiles: the backward produces the weight gradients on the tensor core
        elif precision == PREC_FP32_TC:
            handle.ensure_packed(weights)
        ws = torch.empty(lib.snb_mlp_workspace_bytes(handle.h, m, n_objs, precision), dtype=torch.uint8, device=dev)
        sigma = torch.empty(m, device=dev, dtype=torch.float32)
        rgb = torch.empty(m, 3, device=dev, dtype=torch.float32)
        with on_device(dev):
            check(lib.snb_mlp_fwd(handle.h, precision, ptr(xyz), ptr(viewdir), m, n_objs, ptr(shape_latent), ptr(texture_latent),
                                  ptr(sigma), ptr(rgb), ptr(ws), stream_ptr()), "snb_mlp_fwd")
        ctx.save_for_backward(xyz, viewdir, shape_latent, texture_latent, sigma, ws, *weights)
        ctx.meta = (handle, precision, n_objs, handle._packed_key if precision != PREC["fp32"] else None)
        return sigma, rgb

    @staticmethod
    def backward(ctx, g_sigma, g_rgb):
        lib = _lib.load()
        xyz, viewdir, shape_latent, texture_latent, sigma, ws, *weights = ctx.saved_tensors
        handle, precision, n_objs, packed_key = ctx.meta
        if packed_key is not None and handle._packed_key != packed_key:
            # the weights were re-packed between this graph's forward and its backward (forward, optimizer.step, forward,
            # backward-of-the-first): the masks / activations of the old weights must not meet the W^T images of the new ones
            raise RuntimeError("supnerf_b200: the decoder weights changed between this forward and its backward (bf16 mode keeps ONE "
                               "packed image per handle); run the backward before updating the weights, or use precision='fp32'")
        m = xyz.numel() // 3
        dev = xyz.device
        g_sigma = f32c(g_sigma) if g_sigma is not None else torch.zeros(m, device=dev)
        g_rgb = f32c(g_rgb) if g_rgb is not None else torch.zeros(m, 3, device=dev)
        need = ctx.needs_input_grad
        # the tensor-core backward folds d xyz and d viewdir in one program: when only one of them is wanted the other goes to scratch
        want_pose = need[3] or need[4]
        g_xyz = torch.empty_like(xyz) if want_pose else None
        g_vd = torch.empty_like(viewdir) if want_pose else None
        g_sl = torch.empty_like(shape_latent)
        g_tl = torch.empty_like(texture_latent)
        need_w = any(need[7:])
        gws, gw_arr = None, None
        if need_w:
            gws = [torch.empty_like(w, dtype=torch.float32).contiguous() for w in weights]
            gw_arr = (ctypes.c_void_p * len(gws))(*[g.data_ptr() for g in gws])
        handle.set_weights(weights, saved=True)
        scratch = torch.empty(lib.snb_mlp_bwd_scratch_bytes(handle.h, m, n_objs, precision), dtype=torch.uint8, device=dev)
        with on_device(dev):
            check(lib.snb_mlp_bwd(handle.h, precision, ptr(xyz), ptr(viewdir), m, n_objs, ptr(shape_latent), ptr(texture_latent),
                                  ptr(sigma), ptr(g_sigma), ptr(g_rgb), ptr(ws), ptr(scratch), ptr(g_xyz), ptr(g_vd), ptr(g_sl),
                                  ptr(g_tl), gw_arr, stream_ptr()), "snb_mlp_bwd")
        out_w = tuple(gws) if need_w else tuple(None for _ in weights)
        return (None, None, None, g_xyz if need[3] else None, g_vd if need[4] else None, g_sl if need[5] else None,
                g_tl if need[6] else None) + out_w


def decoder(handle, precision, xyz, viewdir, shape_latent, texture_latent, weights):
    n_objs = shape_latent.shape[0]
    prec = PREC[precision] if isinstance(precision, str) else precision
    m = xyz.shape[0]
    frozen = not (torch.is_grad_enabled() and any(w.requires_grad for w in weights))
    tc_rows = prec == PREC["bf16"] or (frozen and _fp32_tc(handle, prec, None, weights) == PREC_FP32_TC)
    if tc_rows and n_objs == 1 and m % 128 != 0 and m > 0:
        # the tensor-core decoder works on 128-row tiles: pad a single object's rows with copies of its last row (outputs
        # sliced off again, so the copies get zero upstream gradient).  Batched latents must bring tile-aligned row counts.
        pad = 128 - m % 128
        xyz_p = torch.cat([xyz, xyz[-1:].expand(pad, 3)])
        vd_p = torch.cat([viewdir, viewdir[-1:].expand(pad, 3)])
        sigma, rgb = _Decoder.apply(handle, prec, n_objs, xyz_p, vd_p, shape_latent, texture_latent, *weights)
        return sigma[:m], rgb[:m]
    return _Decoder.apply(handle, prec, n_objs, xyz, viewdir, shape_latent, texture_latent, *weights)


# ---------------------------------------------------------------------------------------------------
# fused box render of one object — renderer.py:125-165 (get_rays -> prepare_sampled_rays -> model -> volume_render)
# ---------------------------------------------------------------------------------------------------
_ZEROS = {}


def _zeros_like_cached(dev, n):
    """Read-only zeros (n,) on `dev`, for upstream gradients autograd did not supply (never written by the kernels)."""
    key = (str(dev), int(n))
    z = _ZEROS.get(key)
    if z is None and torch.cuda.is_current_stream_capturing():
        return torch.zeros(n, device=dev, dtype=torch.float32)   # inside a CUDA-graph capture: a graph-private buffer, no synchronisation, not cached
    if z is None:
        if len(_ZEROS) > 64:
            _ZEROS.clear()
        z = torch.zeros(n, device=dev, dtype=torch.float32)
        torch.cuda.current_stream(dev).synchronize()   # one-time: other streams may read it from now on
        _ZEROS[key] = z
    return z


class _RenderBox(torch.autograd.Function):
    """One autograd node for the whole per-object render: two C-ABI calls (snb_render_fwd / snb_render_bwd), every
    intermediate in one workspace tensor.  Differentiable to cam_pose, the latents and (fp32 back end) the weights."""

    @staticmethod
    def forward(ctx, handle, precision, n_samples, flags, geom, px, py, K, c2w, z_steps, jitter, shape_latent,
                texture_latent, *weights):
        lib = _lib.load()
        require_cuda(px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent)
        px, py, K, c2w, z_steps = f32c(px), f32c(py), f32c(K), f32c(c2w), f32c(z_steps)
        jitter = f32c(jitter) if jitter is not None else z_steps   # shell mode: unused by the library
        shape_latent, texture_latent = f32c(shape_latent), f32c(texture_latent)
        n = px.numel()
        dev = px.device
        if geom[0] == "box":      # ("box", half_diag, aabb_half)
            desc = _lib.SnbRenderDesc(n, int(n_samples), int(precision), int(flags), float(geom[1]),
                                      (ctypes.c_float * 3)(*[float(v) for v in geom[2]]), 0, 1.0, 0)
        else:                     # ("shell", obj_diag, shapenet_swap)
            desc = _lib.SnbRenderDesc(n, int(n_samples), int(precision), int(flags), 1.0, (ctypes.c_float * 3)(1.0, 1.0, 1.0), 1,
                                      float(geom[1]), int(bool(geom[2])))
        if weights:   # (frozen weights never enter the autograd node: _render_apply pointed the handle at them already)
            handle.set_weights(weights)
            if precision == PREC["bf16"]:
                handle.ensure_packed(weights)
                if any(ctx.needs_input_grad[13:]):
                    desc.precision = PREC_BF16_TRAIN
        key = (n, int(n_samples), int(desc.precision), int(desc.mode))
        cache = handle.__dict__.setdefault("_render_sizes", {})   # per handle: pure functions of (architecture, N, S, precision, mode)
        sizes = cache.get(key)
        if sizes is None:
            if len(cache) > 512:
                cache.clear()
            sizes = (lib.snb_render_workspace_bytes(handle.h, ctypes.byref(desc)), lib.snb_render_bwd_scratch_bytes(handle.h, ctypes.byref(desc)))
            cache[key] = sizes
        ws = torch.empty(sizes[0], dtype=torch.uint8, device=dev)
        o_rgb = torch.empty(n, 3, device=dev, dtype=torch.float32)
        o_dep = torch.empty(n, device=dev, dtype=torch.float32)
        o_acc = torch.empty(n, device=dev, dtype=torch.float32)
        hit = torch.empty(n, device=dev, dtype=torch.uint8)
        with on_device(dev):
            check(lib.snb_render_fwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(z_steps), ptr(jitter),
                                     ptr(shape_latent), ptr(texture_latent), ptr(o_rgb), ptr(o_dep), ptr(o_acc), ptr(hit), ptr(ws),
                                     stream_ptr()), "snb_render_fwd")
        ctx.save_for_backward(px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent, ws, *weights)
        ctx.meta = (handle, desc, sizes[1], handle._frozen if not weights else None)
        hitb = hit.view(torch.bool)   # 0 / 1 bytes: a zero-copy view
        ctx.mark_non_differentiable(hitb)
        ctx.set_materialize_grads(False)   # unused outputs (depth, the hit mask) arrive as None, not as freshly filled zeros
        return o_rgb, o_dep, o_acc, hitb

    @staticmethod
    def backward(ctx, g_rgb, g_dep, g_acc, _g_hit):
        lib = _lib.load()
        px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent, ws, *weights = ctx.saved_tensors
        handle, desc, scratch_bytes, frozen = ctx.meta
        n = px.numel()
        dev = px.device
        g_rgb = f32c(g_rgb) if g_rgb is not None else _zeros_like_cached(dev, 3 * n)
        g_dep = f32c(g_dep) if g_dep is not None else _zeros_like_cached(dev, n)   # an unused output (e.g. depth): shared zeros
        g_acc = f32c(g_acc) if g_acc is not None else _zeros_like_cached(dev, n)
        need = ctx.needs_input_grad
        g_c2w = torch.empty(3, 4, device=dev, dtype=torch.float32) if need[8] else None
        g_sl = torch.empty_like(shape_latent)
        g_tl = torch.empty_like(texture_latent)
        need_w = any(need[13:])
        gws, gw_arr = None, None
        if need_w:
            gws = [torch.empty_like(w, dtype=torch.float32).contiguous() for w in weights]
            gw_arr = (ctypes.c_void_p * len(gws))(*[g.data_ptr() for g in gws])
        if weights:
            handle.set_weights(weights, saved=True)
        elif frozen is not handle._frozen:   # another weight set was rendered in between: point the handle back at this node's
            handle.use_frozen(frozen, desc.precision)
        scratch = torch.empty(scratch_bytes, dtype=torch.uint8, device=dev)
        with on_device(dev):
            check(lib.snb_render_bwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(z_steps), ptr(jitter),
                                     ptr(shape_latent), ptr(texture_latent), ptr(ws), ptr(g_rgb), ptr(g_dep), ptr(g_acc),
                                     ptr(scratch), ptr(g_c2w), ptr(g_sl), ptr(g_tl), gw_arr, stream_ptr()), "snb_render_bwd")
        out_w = tuple(gws) if need_w else tuple(None for _ in weights)
        return (None,) * 8 + (g_c2w, None, None, g_sl if need[11] else None, g_tl if need[12] else None) + out_w


def _render_apply(handle, prec, n_samples, flags, geom, px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent, weights):
    """Frozen weights (the refine loops: no weight requires grad) stay OUT of the autograd node: 2 x ~30 tensors less to wrap,
    save and return gradients for per object.  The node remembers which weight set it rendered (DecoderHandle.use_frozen)."""
    for w in weights:
        if w.requires_grad:
            break
    else:
        if geom[0] == "box" and os.environ.get("SNB_NO_COMPACT", "0") in ("", "0"):
            prec = _fp32_tc(handle, prec, None, weights)                   # rows compacted on the device: any count
        else:
            prec = _fp32_tc(handle, prec, px.numel() * int(n_samples), weights)    # dense rows
        handle.use_frozen(weights, prec)
        return _RenderBox.apply(handle, prec, n_samples, flags, geom, px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent)
    return _RenderBox.apply(handle, prec, n_samples, flags, geom, px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent, *weights)


def render_box(handle, precision, n_samples, white_bkgd, half_diag, aabb_half, px, py, K, c2w, z_steps, jitter, shape_latent,
               texture_latent, weights):
    """-> rgb (N,3), depth (N,), acc (N,), hit (N,) bool for one object (latents (1,D))."""
    flags = (WHITE_BKGD if white_bkgd else 0) | SIGMA_RELU
    return _render_apply(handle, PREC[precision] if isinstance(precision, str) else precision, n_samples, flags,
                         ("box", half_diag, aabb_half), px, py, K, c2w, z_steps, jitter, shape_latent, texture_latent, weights)


def render_shell(handle, precision, n_samples, obj_diag, shapenet_swap, px, py, K, c2w, z_vals, shape_latent, texture_latent, weights):
    """The utils.py stack (utils.render_rays_v2, utils.py:435-502) for one object: shared sample vector z_vals (S),
    xyz / obj_diag, optional shapenet axis swap, utils.volume_rendering2.  -> rgb (N,3), depth (N,), acc (N,)."""
    rgb, dep, acc, _ = _render_apply(handle, PREC[precision] if isinstance(precision, str) else precision, n_samples, SIGMA_RELU,
                                     ("shell", obj_diag, shapenet_swap), px, py, K, c2w, z_vals, None, shape_latent,
                                     texture_latent, weights)
    return rgb, dep, acc


# ---------------------------------------------------------------------------------------------------
# batched fused box render: B objects in ONE launch set (csrc/render_batch.cu)
# ---------------------------------------------------------------------------------------------------
class _RenderBoxBatch(torch.autograd.Function):
    """Two C-ABI calls (snb_render_batch_fwd / bwd) for the whole batch: ~12 launches forward, ~8 backward whatever B is.
    Frozen weights (the handle points at them, see DecoderHandle.use_frozen), bf16 decoder.  Differentiable to the poses (B,3,4)
    and the latents (B,D)."""

    @staticmethod
    def forward(ctx, handle, n_samples, flags, px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent):
        lib = _lib.load()
        require_cuda(px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent)
        px, py, K, c2w, box, z_steps, jitter = f32c(px), f32c(py), f32c(K), f32c(c2w), f32c(box), f32c(z_steps), f32c(jitter)
        shape_latent, texture_latent = f32c(shape_latent), f32c(texture_latent)
        b, n = px.shape
        dev = px.device
        desc = _lib.SnbBatchDesc(int(b), int(n_samples), int(n), int(flags), 0)
        key = ("batch", b, n, int(n_samples), int(flags) & (FUSED_SAMPLER | BATCH_FP32_TC))
        cache = handle.__dict__.setdefault("_render_sizes", {})
        sizes = cache.get(key)
        if sizes is None:
            sizes = (lib.snb_render_batch_workspace_bytes(handle.h, ctypes.byref(desc)), lib.snb_render_batch_scratch_bytes(handle.h, ctypes.byref(desc)))
            cache[key] = sizes
        ws = torch.empty(sizes[0], dtype=torch.uint8, device=dev)
        o_rgb = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
        o_dep = torch.empty(b, n, device=dev, dtype=torch.float32)
        o_acc = torch.empty(b, n, device=dev, dtype=torch.float32)
        hit = torch.empty(b, n, device=dev, dtype=torch.uint8)
        with on_device(dev):
            check(lib.snb_render_batch_fwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(box), ptr(z_steps), ptr(jitter),
                                           ptr(shape_latent), ptr(texture_latent), ptr(o_rgb), ptr(o_dep), ptr(o_acc), ptr(hit), ptr(ws),
                                           stream_ptr()), "snb_render_batch_fwd")
        ctx.save_for_backward(px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent, ws)
        ctx.meta = (handle, desc, sizes[1], handle._frozen)
        hitb = hit.view(torch.bool)
        ctx.mark_non_differentiable(hitb)
        ctx.set_materialize_grads(False)
        return o_rgb, o_dep, o_acc, hitb

    @staticmethod
    def backward(ctx, g_rgb, g_dep, g_acc, _g_hit):
        lib = _lib.load()
        px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent, ws = ctx.saved_tensors
        handle, desc, scratch_bytes, frozen = ctx.meta
        dev = px.device
        b, n = px.shape
        g_rgb = f32c(g_rgb) if g_rgb is not None else _zeros_like_cached(dev, 3 * b * n)
        g_dep = f32c(g_dep) if g_dep is not None else None     # the library treats NULL as zero
        g_acc = f32c(g_acc) if g_acc is not None else None
        need = ctx.needs_input_grad
        g_c2w = torch.empty(b, 3, 4, device=dev, dtype=torch.float32) if need[6] else None
        g_sl = torch.empty_like(shape_latent)
        g_tl = torch.empty_like(texture_latent)
        if frozen is not handle._frozen:
            handle.use_frozen(frozen, PREC_FP32_TC if desc.flags & BATCH_FP32_TC else PREC["bf16"])
        scratch = torch.empty(scratch_bytes, dtype=torch.uint8, device=dev)
        with on_device(dev):
            check(lib.snb_render_batch_bwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(box), ptr(z_steps), ptr(jitter),
                                           ptr(shape_latent), ptr(texture_latent), ptr(ws), ptr(g_rgb), ptr(g_dep), ptr(g_acc), ptr(scratch),
                                           ptr(g_c2w), ptr(g_sl), ptr(g_tl), stream_ptr()), "snb_render_batch_bwd")
        return (None,) * 6 + (g_c2w, None, None, None, g_sl if need[10] else None, g_tl if need[11] else None)


FUSED_SAMPLER = 4   # SNB_BATCH_FUSED_SAMPLER
BATCH_FP32_TC = 8   # SNB_BATCH_FP32_TC


def render_box_batch(handle, n_samples, white_bkgd, px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent, weights,
                     fused_sampler=False, precision="bf16"):
    """B objects through ONE launch set.  px, py (B,N); K (B,3,3); c2w (B,3,4); box (B,4) = {diag/2, l/diag, w/diag, h/diag}
    (box_constants per object); jitter (B,N,S); latents (B,D).  -> rgb (B,N,3), depth (B,N), acc (B,N), hit (B,N) bool.
    Frozen weights only (refine mode).  precision "bf16" (the two-tile kernels) or "fp32" (the split-precision tensor-core kernels,
    SNB_PREC_FP32_TC: fp32-grade results).  fused_sampler (bf16 only): the decoder's forward computes every row's stratified sample
    from its ray itself (north-star kernel K1: no sampler kernel, no per-row coordinates in HBM on the forward path); bit-identical
    results, measured ~0.7 % slower per forward + backward step than the default, which writes the executed rows' samples once."""
    for w in weights:
        if w.requires_grad:
            raise RuntimeError("render_box_batch: the batched render is the frozen-weight (refine) path; "
                               "model.requires_grad_(False), or render the objects one by one")
    prec = PREC[precision] if isinstance(precision, str) else precision
    flags = (WHITE_BKGD if white_bkgd else 0) | SIGMA_RELU
    if prec == PREC["bf16"]:
        flags |= FUSED_SAMPLER if fused_sampler else 0
        handle.use_frozen(weights, PREC["bf16"])
    else:
        if fused_sampler or not handle.tc_ok or not handle.weights_in_fp16_range(weights):
            raise RuntimeError("render_box_batch(precision='fp32'): runs on the split-precision tensor-core decoder (CodeNeRF family, "
                               "W = 128 or 256, |weights| < 255), without the fused sampler; render the objects one by one otherwise")
        flags |= BATCH_FP32_TC
        handle.use_frozen(weights, PREC_FP32_TC)
    return _RenderBoxBatch.apply(handle, n_samples, flags, px, py, K, c2w, box, z_steps, jitter, shape_latent, texture_latent)


class _RenderShellBatch(torch.autograd.Function):
    """utils.render_rays_v2's stack (utils.py:435-502) for B objects: two C-ABI calls (snb_render_shell_batch_fwd / bwd), ~5 launches
    forward and ~7 backward whatever B is.  Frozen weights.  Differentiable to the poses (B,3,4) and the latents (B,D)."""

    @staticmethod
    def forward(ctx, handle, precision, n_samples, swap, px, py, K, c2w, z, obj_diag, shape_latent, texture_latent):
        lib = _lib.load()
        require_cuda(px, py, K, c2w, z, obj_diag, shape_latent, texture_latent)
        px, py, K, c2w, z, obj_diag = f32c(px), f32c(py), f32c(K), f32c(c2w), f32c(z), f32c(obj_diag)
        shape_latent, texture_latent = f32c(shape_latent), f32c(texture_latent)
        b, n = px.shape
        dev = px.device
        desc = _lib.SnbShellBatchDesc(int(b), int(n_samples), int(n), int(precision), SIGMA_RELU, int(bool(swap)), 0)
        key = ("shell_batch", b, n, int(n_samples), int(precision))
        cache = handle.__dict__.setdefault("_render_sizes", {})
        sizes = cache.get(key)
        if sizes is None:
            sizes = (lib.snb_render_shell_batch_workspace_bytes(handle.h, ctypes.byref(desc)),
                     lib.snb_render_shell_batch_scratch_bytes(handle.h, ctypes.byref(desc)))
            cache[key] = sizes
        ws = torch.empty(sizes[0], dtype=torch.uint8, device=dev)
        o_rgb = torch.empty(b, n, 3, device=dev, dtype=torch.float32)
        o_dep = torch.empty(b, n, device=dev, dtype=torch.float32)
        o_acc = torch.empty(b, n, device=dev, dtype=torch.float32)
        with on_device(dev):
            check(lib.snb_render_shell_batch_fwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(z), ptr(obj_diag),
                                                 ptr(shape_latent), ptr(texture_latent), ptr(o_rgb), ptr(o_dep), ptr(o_acc), ptr(ws),
                                                 stream_ptr()), "snb_render_shell_batch_fwd")
        ctx.save_for_backward(px, py, K, c2w, z, obj_diag, shape_latent, texture_latent, ws)
        ctx.meta = (handle, desc, sizes[1], handle._frozen)
        ctx.set_materialize_grads(False)
        return o_rgb, o_dep, o_acc

    @staticmethod
    def backward(ctx, g_rgb, g_dep, g_acc):
        lib = _lib.load()
        px, py, K, c2w, z, obj_diag, shape_latent, texture_latent, ws = ctx.saved_tensors
        handle, desc, scratch_bytes, frozen = ctx.meta
        dev = px.device
        b, n = px.shape
        g_rgb = f32c(g_rgb) if g_rgb is not None else _zeros_like_cached(dev, 3 * b * n)
        g_dep = f32c(g_dep) if g_dep is not None else _zeros_like_cached(dev, b * n)
        g_acc = f32c(g_acc) if g_acc is not None else _zeros_like_cached(dev, b * n)
        need = ctx.needs_input_grad
        g_c2w = torch.empty(b, 3, 4, device=dev, dtype=torch.float32) if need[7] else None
        g_sl = torch.empty_like(shape_latent)
        g_tl = torch.empty_like(texture_latent)
        if frozen is not handle._frozen:
            handle.use_frozen(frozen, desc.precision)
        scratch = torch.empty(scratch_bytes, dtype=torch.uint8, device=dev)
        with on_device(dev):
            check(lib.snb_render_shell_batch_bwd(handle.h, ctypes.byref(desc), ptr(px), ptr(py), ptr(K), ptr(c2w), ptr(z), ptr(obj_diag),
                                                 ptr(shape_latent), ptr(texture_latent), ptr(ws), ptr(g_rgb), ptr(g_dep), ptr(g_acc),
                                                 ptr(scratch), ptr(g_c2w), ptr(g_sl), ptr(g_tl), stream_ptr()), "snb_render_shell_batch_bwd")
        return (None,) * 7 + (g_c2w, None, None, g_sl if need[10] else None, g_tl if need[11] else None)


def render_shell_batch(handle, precision, n_samples, shapenet_swap, px, py, K, c2w, z_vals, obj_diag, shape_latent, texture_latent, weights):
    """utils.render_rays_v2 (utils.py:435-502) for B objects through ONE launch set.  px, py (B,N); K (B,3,3); c2w (B,3,4); z_vals (B,S)
    every object's shared sample vector; obj_diag (B) on the device; latents (B,D).  -> rgb (B,N,3), depth (B,N), acc (B,N).
    Frozen weights only (the refine loops); the bf16 decoder needs N * S to be a multiple of 128."""
    for w in weights:
        if w.requires_grad:
            raise RuntimeError("render_shell_batch: the batched render is the frozen-weight (refine) path; "
                               "model.requires_grad_(False), or render the objects one by one")
    prec = _fp32_tc(handle, PREC[precision] if isinstance(precision, str) else precision, px.shape[1] * int(n_samples), weights)
    handle.use_frozen(weights, prec)
    return _RenderShellBatch.apply(handle, prec, n_samples, shapenet_swap, px, py, K, c2w, z_vals, obj_diag, shape_latent, texture_latent)


def box_constants(obj_sz):
    """renderer.py:92-100: diag and the AABB half extents (l,w,h)/diag, rounded to float32 on the host."""
    obj_sz = np.asarray(obj_sz)
    diag = np.linalg.norm(obj_sz).astype(np.float32)
    w, l, h = obj_sz
    half = np.asarray([l / diag, w / diag, h / diag]).astype(np.float32)
    return diag, half
