"""CPU oracle for the SUP-NeRF object-centric volumetric render hot path.

TEST INFRASTRUCTURE ONLY.  This module is a from-scratch restatement (torch CPU ops, dtype-generic,
plus numpy for the integer/bool part) of what the reference computes on the hot path; it is the
checker for the CUDA kernels.  Only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it.  The product package ``supnerf_b200`` never
imports it and has no CPU fallback.

Parity status: PINNED.  Every function here is checked against outputs of the unmodified reference
(``/root/reference/src/{renderer,utils,model_*}.py`` imported in the build container by
``tools/make_golden.py``); the resulting fixtures live in ``tests/golden/`` and are re-checked by
``tests/test_oracle_golden.py`` (runs on CPU, does not need ``/root/reference``).

Citations are ``file:line`` into ``/root/reference/src``.

Stated divergence: ``composite`` at S = 1.  The reference builds the last sample's 1e10 delta from ``deltas[..., :1]``, which is
empty when a ray has one sample, so it cannot composite S = 1 at all; here the single sample is the last one (delta 1e10), as in
the library's compositing (composite.cuh) and in ``composite_backward_closed_form``.  Every S >= 2 is unchanged.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

Tensor = torch.Tensor


# --------------------------------------------------------------------------------------------------
# a1. ray generation
# --------------------------------------------------------------------------------------------------
def pixel_grid(roi: Sequence[int], uv_steps: Optional[Sequence[int]] = None) -> Tuple[Tensor, Tensor]:
    """Pixel coordinates of the roi, row-major (v outer, u inner).  utils.py:121-128.

    ``torch.linspace`` is kept (not re-derived) because its fp32 rounding (symmetric two-sided formula)
    is part of the reference's result."""
    x0, y0, x1, y1 = [int(v) for v in roi]
    if uv_steps is not None:
        us = torch.linspace(x0, x1 - 1, int(uv_steps[0]))
        vs = torch.linspace(y0, y1 - 1, int(uv_steps[1]))
    else:
        us = torch.linspace(x0, x1 - 1, x1 - x0)
        vs = torch.linspace(y0, y1 - 1, y1 - y0)
    # meshgrid(ij).t() == v outer / u inner
    i = us.unsqueeze(0).expand(vs.numel(), us.numel())
    j = vs.unsqueeze(1).expand(vs.numel(), us.numel())
    return i, j


def rays_from_pixels(K: Tensor, c2w: Tensor, i: Tensor, j: Tensor) -> Tuple[Tensor, Tensor]:
    """utils.py:130-135 (also :146-151): back-project, rotate, normalise; origin = c2w[:, 3]."""
    cx, cy, fx, fy = K[0, 2], K[1, 2], K[0, 0], K[1, 1]
    dirs = torch.stack([(i - cx) / fx, (j - cy) / fy, torch.ones_like(i)], -1)
    rays_d = torch.sum(dirs[..., None, :].type_as(c2w) * c2w[..., :3, :3], -1)
    viewdirs = rays_d / torch.norm(rays_d, dim=-1, keepdim=True)
    rays_o = c2w[..., :3, -1].expand(rays_d.shape)
    return rays_o.reshape(-1, 3), viewdirs.reshape(-1, 3)


def get_rays(K: Tensor, c2w: Tensor, roi, uv_steps=None) -> Tuple[Tensor, Tensor]:
    """utils.py:107-135."""
    i, j = pixel_grid(roi, uv_steps)
    return rays_from_pixels(K, c2w, i, j)


def get_rays_specified(K: Tensor, c2w: Tensor, x_vec: np.ndarray, y_vec: np.ndarray):
    """utils.py:138-151."""
    i = torch.from_numpy(np.asarray(x_vec)).t()
    j = torch.from_numpy(np.asarray(y_vec)).t()
    return rays_from_pixels(K, c2w, i, j)


# --------------------------------------------------------------------------------------------------
# a2. slab test
# --------------------------------------------------------------------------------------------------
def ray_box_intersection_np(ray_o: np.ndarray, ray_d: np.ndarray, aabb_min=None, aabb_max=None):
    """utils.py:236-280, numpy, same IEEE op order (reciprocal; sub then mul; min/max; two compares)."""
    if aabb_min is None:
        aabb_min = np.ones_like(ray_o) * -1.0
    if aabb_max is None:
        aabb_max = np.ones_like(ray_o)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv_d = np.reciprocal(ray_d)
        t_min = (aabb_min - ray_o) * inv_d
        t_max = (aabb_max - ray_o) * inv_d
    t0 = np.minimum(t_min, t_max)
    t1 = np.maximum(t_min, t_max)
    t_near = np.maximum(np.maximum(t0[..., 0], t0[..., 1]), t0[..., 2])
    t_far = np.minimum(np.minimum(t1[..., 0], t1[..., 1]), t1[..., 2])
    hit = t_far > t_near
    with np.errstate(invalid="ignore"):
        hit = np.logical_and(hit, (t_far * hit) > 0)
    return t_near, t_far, hit


def ray_box_intersection(ray_o: Tensor, ray_d: Tensor, aabb_min: Tensor, aabb_max: Tensor):
    """utils.py:283-327 — returns the *uncompacted* (t_near, t_far, hit); the reference's
    ``t_near[hit]`` compaction is applied by the caller."""
    inv_d = torch.reciprocal(ray_d)
    t_min = (aabb_min - ray_o) * inv_d
    t_max = (aabb_max - ray_o) * inv_d
    t0 = torch.minimum(t_min, t_max)
    t1 = torch.maximum(t_min, t_max)
    t_near = torch.maximum(torch.maximum(t0[..., 0], t0[..., 1]), t0[..., 2])
    t_far = torch.minimum(torch.minimum(t1[..., 0], t1[..., 1]), t1[..., 2])
    hit = t_far > t_near
    hit = torch.logical_and(hit, (t_far * hit) > 0)
    return t_near, t_far, hit


# --------------------------------------------------------------------------------------------------
# a3/a4. samplers
# --------------------------------------------------------------------------------------------------
def box_constants(obj_sz: np.ndarray) -> Tuple[np.float32, np.ndarray]:
    """renderer.py:92-100 — diag and AABB half extents (l, w, h)/diag, rounded to float32 on the host."""
    obj_sz = np.asarray(obj_sz)
    diag = np.linalg.norm(obj_sz).astype(np.float32)
    w, l, h = obj_sz
    half = np.asarray([l / diag, w / diag, h / diag]).astype(np.float32)
    return diag, half


def stratified_z(near: Tensor, far: Tensor, n_samples: int, jitter: Tensor) -> Tensor:
    """renderer.py:27-41 ≡ utils.py:170-184.  ``jitter`` is the U[0,1) draw of ``torch.rand_like``
    (shape (N,S)); near/far are (N,1)."""
    step = 1.0 / n_samples
    z_steps = torch.linspace(0, 1 - step, n_samples, device=near.device)
    z_steps = z_steps.unsqueeze(0).repeat(near.shape[0], 1).to(near.dtype)
    z_steps = z_steps + jitter * step
    return near * (1 - z_steps) + far * z_steps


def prepare_sampled_rays(rays_o: Tensor, viewdir: Tensor, obj_sz: np.ndarray, n_samples: int, jitter: Tensor):
    """renderer.py:91-115.  Returns xyz (N,S,3), viewdir (N,S,3), z_vals (N,S), intersect (N,) bool."""
    diag, half = box_constants(obj_sz)
    N = rays_o.shape[0]
    half_t = torch.from_numpy(half).to(rays_o.device)
    aabb_max = half_t.reshape(1, 3).repeat(N, 1)
    aabb_min = -aabb_max
    o_n = rays_o / (diag / 2)
    t_near, t_far, hit = ray_box_intersection(o_n, viewdir, aabb_min.to(o_n.dtype), aabb_max.to(o_n.dtype))
    minus1 = torch.full_like(t_near, -1)
    near = torch.where(hit, t_near, minus1)  # == index_put of the compacted values (renderer.py:105-107)
    far = torch.where(hit, t_far, minus1)
    z = stratified_z(near[:, None], far[:, None], n_samples, jitter)
    xyz = o_n[:, None, :] + z[:, :, None] * viewdir[:, None, :]
    vd = viewdir.unsqueeze(-2).repeat(1, n_samples, 1)
    z_vals = torch.norm((xyz - o_n[:, None, :]) * (diag / 2), p=2, dim=-1)
    return xyz, vd, z_vals, hit


def shell_bounds(cam_pose: Tensor, obj_diag: float) -> Tuple[float, float]:
    """utils.py:468-469: near/far = ‖t‖ ∓ diag/2 as detached python floats."""
    n = np.linalg.norm(cam_pose.detach()[:, -1].tolist())
    return n - obj_diag / 2, n + obj_diag / 2


def sample_from_rays_shell(ro: Tensor, vd: Tensor, near: float, far: float, n_samples: int, jitter: Optional[Tensor]):
    """utils.py:154-167.  ``jitter`` is the CPU ``torch.rand(N_samples)`` draw (None ⇒ z_fixed)."""
    if jitter is None:
        z_vals = torch.linspace(near, far, n_samples).type_as(ro)
    else:
        dist = (far - near) / (2 * n_samples)
        z_vals = torch.linspace(near + dist, far - dist, n_samples).type_as(ro)
        z_vals = z_vals + (jitter * (far - near) / (2 * n_samples)).type_as(ro)
    xyz = ro.unsqueeze(-2) + vd.unsqueeze(-2) * z_vals.unsqueeze(-1)
    vd = vd.unsqueeze(-2).repeat(1, n_samples, 1)
    return xyz, vd, z_vals


def shapenet_swap(x: Tensor) -> Tensor:
    """(x, y, z) -> (-y, x, z); utils.py:491-495, renderer.py:459-463."""
    return torch.stack([-x[..., 1], x[..., 0], x[..., 2]], -1)


# --------------------------------------------------------------------------------------------------
# a5. positional encoding
# --------------------------------------------------------------------------------------------------
def positional_encoding(x: Tensor, degree: int) -> Tensor:
    """model_codenerf.py:4-10: [x, sin(2^i x) for i<deg (3-wide blocks), cos(2^i x) for i<deg]."""
    y = torch.cat([2.0 ** i * x for i in range(degree)], -1)
    return torch.cat([x, torch.sin(y), torch.cos(y)], -1)


# --------------------------------------------------------------------------------------------------
# a6/a7. decoders.  Weights are addressed by the reference's state_dict keys (the weight ABI).
# --------------------------------------------------------------------------------------------------
def _lin(sd: Dict[str, Tensor], name: str, x: Tensor) -> Tensor:
    return torch.nn.functional.linear(x, sd[name + ".weight"], sd[name + ".bias"])


def decoder_blocks(sd: Dict[str, Tensor]) -> Tuple[int, int]:
    bs = sum(1 for k in sd if k.startswith("shape_layer_") and k.endswith(".0.weight"))
    bt = sum(1 for k in sd if k.startswith("texture_layer_") and k.endswith(".0.weight"))
    return bs, bt


def codenerf_decoder(sd: Dict[str, Tensor], xyz: Tensor, viewdir: Tensor, shape_latent: Tensor,
                     texture_latent: Tensor, num_xyz_freq: int = 10, num_dir_freq: int = 4,
                     return_acts: bool = False):
    """model_codenerf.py:39-63 ≡ model_autorf.py:226-250 ≡ model_supnerf.py:241-269.

    xyz/viewdir (N,S,3); latents (B,D); object b owns rays [b*N/B, (b+1)*N/B)."""
    bs, bt = decoder_blocks(sd)
    x = positional_encoding(xyz, num_xyz_freq)
    v = positional_encoding(viewdir, num_dir_freq)
    B = shape_latent.shape[0]
    ppi = int(xyz.shape[0] / B)
    sl = shape_latent.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    tl = texture_latent.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    acts: List[Tensor] = []
    y = torch.relu(_lin(sd, "encoding_xyz.0", x))
    acts.append(y)
    for j in range(1, bs + 1):
        z = torch.relu(_lin(sd, f"shape_latent_layer_{j}.0", sl))
        y = torch.relu(_lin(sd, f"shape_layer_{j}.0", y + z))
        acts.append(y)
    y = _lin(sd, "encoding_shape", y)
    acts.append(y)
    sigmas = torch.nn.functional.softplus(_lin(sd, "sigma.0", y))
    y = torch.relu(_lin(sd, "encoding_viewdir.0", torch.cat([y, v], -1)))
    acts.append(y)
    for j in range(1, bt + 1):
        z = torch.relu(_lin(sd, f"texture_latent_layer_{j}.0", tl))
        y = torch.relu(_lin(sd, f"texture_layer_{j}.0", y + z))
        acts.append(y)
    h = torch.relu(_lin(sd, "rgb.0", y))
    acts.append(h)
    rgbs = _lin(sd, "rgb.2", h)
    if return_acts:
        return sigmas, rgbs, acts
    return sigmas, rgbs


class _RoundBF16(torch.autograd.Function):
    """Round to bf16 in the forward AND the backward pass (what a bf16 MMA operand sees in either direction)."""

    @staticmethod
    def forward(ctx, x):
        return x.bfloat16().to(x.dtype)

    @staticmethod
    def backward(ctx, g):
        return g.bfloat16().to(g.dtype)


def codenerf_decoder_bf16(sd: Dict[str, Tensor], xyz: Tensor, viewdir: Tensor, shape_latent: Tensor,
                          texture_latent: Tensor, num_xyz_freq: int = 10, num_dir_freq: int = 4):
    """Restatement of the SNB_PREC_BF16 mode's arithmetic (supnerf_b200/csrc/mlp_tc.cu), NOT of the reference: the
    same decoder as ``codenerf_decoder`` with every tensor-core operand rounded to bf16 where the kernel rounds it —
    the weight matrices of the 63/256/283-input layers and rgb.0, the encodings, each layer's A operand (the post-ReLU
    activation; the per-object latent vector enters as an fp32 effective bias  z W^T + b) and, in the backward pass, each
    pre-activation gradient.  Biases,
    latent layers, the sigma and rgb.2 heads and all accumulation stay fp32.  Used to separate "the kernel implements
    its stated rounding" (tight) from "bf16 rounding vs the fp32 reference" (the 2e-2 budget)."""
    rb = _RoundBF16.apply
    bs, bt = decoder_blocks(sd)

    def mm(name, x):
        return torch.nn.functional.linear(x, sd[name + ".weight"].bfloat16().to(x.dtype), sd[name + ".bias"])

    x = rb(positional_encoding(xyz, num_xyz_freq))
    v = rb(positional_encoding(viewdir, num_dir_freq))
    B = shape_latent.shape[0]
    ppi = int(xyz.shape[0] / B)
    sl = shape_latent.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    tl = texture_latent.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    def mm_lat(name, y, z):
        # (y + z) W^T + b  evaluated as  bf16(y) bf16(W)^T + (z W^T + b): the latent term is a per-object fp32 bias
        w = sd[name + ".weight"]
        return torch.nn.functional.linear(rb(y), w.bfloat16().to(y.dtype)) + torch.nn.functional.linear(z, w, sd[name + ".bias"])

    y = torch.relu(mm("encoding_xyz.0", x))
    for j in range(1, bs + 1):
        z = torch.relu(_lin(sd, f"shape_latent_layer_{j}.0", sl))
        y = torch.relu(mm_lat(f"shape_layer_{j}.0", y, z))
    e = mm("encoding_shape", rb(y))
    sigmas = torch.nn.functional.softplus(_lin(sd, "sigma.0", e))
    y = torch.relu(mm("encoding_viewdir.0", torch.cat([rb(e), v], -1)))
    for j in range(1, bt + 1):
        z = torch.relu(_lin(sd, f"texture_latent_layer_{j}.0", tl))
        y = torch.relu(mm_lat(f"texture_layer_{j}.0", y, z))
    h = torch.relu(mm("rgb.0", rb(y)))
    rgbs = _lin(sd, "rgb.2", h)
    return sigmas, rgbs


def autorf_decoder(sd: Dict[str, Tensor], xyz: Tensor, viewdir: Tensor, shape_feat: Tensor, texture_feat: Tensor,
                   shape_blocks: int = 5, texture_blocks: int = 5, num_xyz_freq: int = 10, num_dir_freq: int = 4):
    """model_autorf.py:156-186 (the non-mix AutoRF decoder, W = latent_dim)."""
    x = positional_encoding(xyz, num_xyz_freq)
    pos = torch.relu(_lin(sd, "encoding_xyz.0", x))
    v = positional_encoding(viewdir, num_dir_freq)
    B = shape_feat.shape[0]
    ppi = int(xyz.shape[0] / B)
    sf = shape_feat.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    tf = texture_feat.unsqueeze(1).repeat((1, ppi, 1)).reshape((ppi * B, 1, -1))
    for j in range(shape_blocks - 1):
        sf = (sf + pos) / 2
        sf = torch.relu(_lin(sd, f"shape_layer_{j}.0", sf))
    sigmas = torch.nn.functional.softplus(_lin(sd, "sigma.0", (sf + pos) / 2))
    for j in range(texture_blocks - 2):
        tf = (tf + pos) / 2
        tf = torch.relu(_lin(sd, f"texture_layer_{j}.0", tf))
    tf = (tf + sf + pos) / 3
    tf = torch.cat([tf, v], dim=-1)
    tf = torch.relu(_lin(sd, f"texture_layer_{texture_blocks - 2}.0", tf))
    tf = (tf + pos) / 2
    tf = torch.cat([tf, v], dim=-1)
    rgbs = torch.sigmoid(_lin(sd, "rgb.0", tf))
    return sigmas, rgbs


from supnerf_b200.synthetic import (NUSC_K, WLH_MEAN, WLH_STD, init_autorf_state, init_codenerf_state,  # noqa: E402,F401
                                    synthetic_latents, synthetic_object)


# --------------------------------------------------------------------------------------------------
# a8. compositing
# --------------------------------------------------------------------------------------------------
def composite(sigmas: Tensor, rgbs: Tensor, z_vals: Tensor, white_bkgd: bool, use_relu: bool = True):
    """renderer.py:43-65 / :355-379 (per-ray z_vals (N,S)); utils.py:202-217 (z_vals (S,));
    utils.py:220-233 (sigmas (B,n,S), z_vals (B,S)); utils.py:187-199 (``use_relu=False``).

    sigmas (...,S), rgbs (...,S,3), z_vals broadcastable to sigmas.  Returns rgb (...,3), depth (...),
    acc (...) with acc = transmittance *before* the last sample."""
    if z_vals.dim() == 1:  # one shared vector (S,)
        z = z_vals.expand_as(sigmas)
    elif sigmas.dim() == 3 and z_vals.dim() == 2:  # (B,S) against (B,n,S)
        z = z_vals.unsqueeze(1).expand_as(sigmas)
    else:
        z = z_vals
    deltas = z[..., 1:] - z[..., :-1]
    # (z[..., :1], not the reference's deltas[..., :1]: the same column for S >= 2, and S = 1 works -- see the module docstring)
    deltas = torch.cat([deltas, torch.ones_like(z[..., :1]) * 1e10], -1)
    s = torch.relu(sigmas) if use_relu else sigmas
    alphas = 1 - torch.exp(-s * deltas)
    trans = 1 - alphas + 1e-10
    transmittance = torch.cat([torch.ones_like(trans[..., :1]), trans], -1)
    accum = torch.cumprod(transmittance, -1)[..., :-1]
    weights = alphas * accum
    rgb = torch.sum(weights.unsqueeze(-1) * rgbs, -2)
    depth = torch.sum(weights * z, -1)
    if white_bkgd:
        rgb = rgb + 1 - weights.sum(dim=-1).unsqueeze(-1)
    return rgb, depth, accum[..., -1]


def composite_backward_closed_form(sigmas, rgbs, z_vals, g_rgb, g_depth, g_acc, white_bkgd: bool, use_relu=True):
    """Closed-form gradient of ``composite`` for per-ray z_vals (N,S) — the spec of kernel K3b
    (SURVEY §8(a) row a8); checked against autograd in tests."""
    N, S = sigmas.shape
    z = z_vals
    deltas = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1)
    s = torch.relu(sigmas) if use_relu else sigmas
    e = torch.exp(-s * deltas)
    alphas = 1 - e
    t = 1 - alphas + 1e-10
    T = torch.cumprod(torch.cat([torch.ones_like(t[:, :1]), t], -1), -1)[:, :-1]
    w = alphas * T
    A = T[:, -1]
    gw = (g_rgb[:, None, :] * rgbs).sum(-1) + g_depth[:, None] * z
    if white_bkgd:
        gw = gw - g_rgb.sum(-1, keepdim=True)
    g_c = w[..., None] * g_rgb[:, None, :]
    gww = gw * w
    suffix = torch.flip(torch.cumsum(torch.flip(gww, [-1]), -1), [-1]) - gww  # sum_{k>j}
    tail = torch.ones_like(suffix)
    tail[:, -1] = 0
    g_t = (suffix + tail * (g_acc * A)[:, None]) / t
    g_alpha = gw * T - g_t
    mask = (sigmas > 0).to(sigmas.dtype) if use_relu else torch.ones_like(sigmas)
    g_sigma = g_alpha * deltas * e * mask
    g_delta = g_alpha * s * e
    g_delta[:, -1] = 0
    g_z = w * g_depth[:, None]
    g_z[:, 1:] += g_delta[:, :-1]
    g_z -= g_delta
    return g_sigma, g_c, g_z


# --------------------------------------------------------------------------------------------------
# a9. drivers (one object / view)
# --------------------------------------------------------------------------------------------------
def render_rays_box(sd, K, cam_pose, obj_sz, roi, im_sz, n_samples, shapecode, texturecode, jitter,
                    white_bkgd=True, ray_ids=None, decoder=codenerf_decoder):
    """NeRFRenderer.render_rays, renderer.py:117-167, minus the target resize (targets are inputs,
    not renders).  ``jitter`` (N,S) replaces torch.rand_like; ``ray_ids`` replaces the numpy
    permutation (renderer.py:139-146).  ``decoder``: codenerf_decoder, or codenerf_decoder_bf16 for the bf16 mode's rounding."""
    rays_o, viewdir = get_rays(K, cam_pose, roi, uv_steps=[im_sz, im_sz])
    if ray_ids is not None:
        rays_o, viewdir = rays_o[ray_ids], viewdir[ray_ids]
    xyz, vd, z_vals, hit = prepare_sampled_rays(rays_o, viewdir, obj_sz, n_samples, jitter)
    sigmas, rgbs = decoder(sd, xyz, vd, shapecode, texturecode)
    rgb, depth, acc = composite(sigmas.squeeze(-1), rgbs, z_vals, white_bkgd)
    return rgb, depth, acc, hit


def render_rays_shell(sd, K, cam_pose, obj_diag, roi, im_sz, n_samples, shapecode, texturecode, jitter,
                      shapenet_obj_cood=True, ray_ids=None, decoder=codenerf_decoder):
    """utils.render_rays_v2, utils.py:435-502 (sym_aug / kitti2nusc off), targets excluded.  ``decoder`` as in render_rays_box."""
    rays_o, viewdir = get_rays(K, cam_pose, roi, uv_steps=[im_sz, im_sz])
    if ray_ids is not None:
        rays_o, viewdir = rays_o[ray_ids], viewdir[ray_ids]
    obj_diag = float(obj_diag)  # np.float32 scalar in the reference; exactly representable
    near, far = shell_bounds(cam_pose.detach(), obj_diag)
    xyz, vd, z_vals = sample_from_rays_shell(rays_o, viewdir, near, far, n_samples, jitter)
    xyz = xyz / obj_diag
    if shapenet_obj_cood:
        xyz = shapenet_swap(xyz)
        vd = shapenet_swap(vd)
    sigmas, rgbs = decoder(sd, xyz, vd, shapecode, texturecode)
    rgb, depth, acc = composite(sigmas.squeeze(-1), rgbs, z_vals, white_bkgd=False)
    return rgb, depth, acc


def refine_losses(rgb_rays, acc_rays, rgb_tgt, occ_pixels, loss_occ_coef=0.1):
    """optimizer_nuscenes.py:729-736: masked MSE + exponential occupancy loss."""
    den = torch.sum(torch.abs(occ_pixels)) + 1e-9
    loss_rgb = torch.sum((rgb_rays - rgb_tgt) ** 2 * torch.abs(occ_pixels)) / den
    loss_occ = torch.sum(torch.exp(-occ_pixels * (0.5 - acc_rays.unsqueeze(-1))) * torch.abs(occ_pixels)) / den
    return loss_rgb + loss_occ_coef * loss_occ, loss_rgb, loss_occ


# --------------------------------------------------------------------------------------------------
# next row (SURVEY 8f rank 4): multi-object scene compositor, merge step
# --------------------------------------------------------------------------------------------------
def merge_objects(z_vals: Tensor, sigmas: Tensor, rgbs: Tensor):
    """scripts/demo.py:560-567: sort every ray's Nb*S depths, ``searchsorted`` the originals into them and scatter sigma / rgb
    to those slots.  Ties collide on one slot; the sequential CPU ``scatter_`` keeps the LAST element in index order and
    leaves the other slots of the tie group zero (pinned by tests/golden/scene_merge.npz, produced by executing those very
    source lines).  z_vals, sigmas (R,K); rgbs (R,K,3) -> z_sort, sigmas_sort, rgbs_sort, z_args."""
    z_sort = torch.sort(z_vals, 1).values
    z_args = torch.searchsorted(z_sort, z_vals.contiguous())
    rgbs_sort = torch.zeros_like(rgbs).scatter_(1, z_args[:, :, None].repeat(1, 1, 3), rgbs)
    sigmas_sort = torch.zeros_like(sigmas).scatter_(1, z_args, sigmas)
    return z_sort, sigmas_sort, rgbs_sort, z_args

