#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference.

Runs only in the build container (needs /root/reference).  It imports the reference's own modules
(renderer.py, utils.py, model_*.py) read-only with stub modules for the absent, off-path
dependencies (matplotlib), executes the hot-path functions on seeded synthetic inputs, and stores
inputs + outputs + gradients as small .npz files.  tests/test_oracle_golden.py pins oracle/oracle.py
against them; the -m gpu tests pin the CUDA kernels against the same files.

Usage: python tools/make_golden.py            (rewrites tests/golden/*.npz)
"""
import hashlib
import math
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/src"
OUT = os.path.join(ROOT, "tests", "golden")

sys.modules.setdefault("matplotlib", types.ModuleType("matplotlib"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import model_autorf  # noqa: E402  (reference)
import model_codenerf  # noqa: E402
import model_supnerf  # noqa: E402
import renderer as ref_renderer  # noqa: E402
import utils as ref_utils  # noqa: E402

from oracle import oracle  # noqa: E402

SAMPLE_MAX = 8192   # arrays save() samples keep at most this many elements: every fixture stays under 1 MB


def state_hash(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def npy(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def sample_stride(a):
    """Smallest stride that keeps at most SAMPLE_MAX elements of the flattened array and is coprime with its last dimension, so
    that the sample visits every row and every column."""
    s = -(-a.size // SAMPLE_MAX)
    while math.gcd(s, a.shape[-1]) != 1:
        s += 1
    return s


def save(name, sample=(), **arrs):
    """Arrays whose key starts with a prefix in `sample` and that hold more than SAMPLE_MAX elements are stored as every
    sample_stride()-th element of their flattened form, beside their shape, the stride and max|.| of the whole array
    (tests/conftest.py:load_golden reads them back as `Sampled`)."""
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    out = {}
    for k, v in arrs.items():
        a = npy(v)
        if k.startswith(tuple(sample)) and a.size > SAMPLE_MAX:
            s = sample_stride(a)
            out.update({k: a.reshape(-1)[::s].copy(), k + "@shape": np.asarray(a.shape, np.int64), k + "@stride": np.int64(s),
                        k + "@absmax": np.float64(np.abs(a.astype(np.float64)).max())})
        else:
            out[k] = a
    np.savez_compressed(path, **out)
    print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


def losses(rgb, acc, tgt, occ):
    return oracle.refine_losses(rgb, acc, tgt, occ)[0]


# ---------------------------------------------------------------------------------------------------
def golden_stages():
    """Stage-level vectors: ray gen, slab test (edge cases), stratified z, PE, compositing variants."""
    torch.manual_seed(7)
    np.random.seed(7)
    obj = oracle.synthetic_object(3, im_sz=12)
    K, c2w, roi = obj["K"], obj["cam_pose"], obj["roi"]
    ro, vd = ref_utils.get_rays(K, c2w, roi, uv_steps=[12, 12])
    ro_full, vd_full = ref_utils.get_rays(K, c2w, torch.tensor([100, 50, 109, 57], dtype=torch.int32))
    xv = np.asarray([0, 3, 5, 7], dtype=np.int64)
    yv = np.asarray([1, 2, 4, 6], dtype=np.int64)
    ro_s, vd_s = ref_utils.get_rays_specified(K, c2w, xv + roi[0].numpy(), yv + roi[1].numpy())

    # slab-test edge cases in the normalised box frame
    half = np.asarray([0.9, 0.4, 0.3], dtype=np.float32)
    o = [[-3, 0, 0], [-3, 0, 0], [0, 0, 0], [-3, 0.4, 0], [-3, 0.41, 0], [3, 0, 0], [-3, 0, 0], [0.9, 0, 0],
         [-3, 0.39999, 0.2999], [2, 2, 2]]
    d = [[1, 0, 0], [-1, 0, 0], [0.6, 0.8, 0], [1, 0, 0], [1, 0, 0], [1, 0, 0], [0, 1, 0], [1, 0, 0],
         [1, 0, 0], [-0.57735026, -0.57735026, -0.57735026]]
    rnd_o = (np.random.randn(200, 3) * 2).astype(np.float32)
    rnd_d = np.random.randn(200, 3).astype(np.float32)
    rnd_d /= np.linalg.norm(rnd_d, axis=1, keepdims=True)
    eo = np.concatenate([np.asarray(o, np.float32), rnd_o])
    ed = np.concatenate([np.asarray(d, np.float32), rnd_d])
    amin = np.repeat(-half[None], eo.shape[0], 0)
    amax = np.repeat(half[None], eo.shape[0], 0)
    with np.errstate(all="ignore"):
        zi_np, zo_np, hit_np = ref_utils.ray_box_intersection(eo, ed, amin, amax)
    zi_t, zo_t, hit_t = ref_utils.ray_box_intersection_tensor(torch.from_numpy(eo), torch.from_numpy(ed),
                                                             torch.from_numpy(amin), torch.from_numpy(amax))
    # default unit box
    zi_u, zo_u, hit_u = ref_utils.ray_box_intersection_tensor(torch.from_numpy(eo), torch.from_numpy(ed))

    # stratified z
    S = 16
    rays = torch.cat([torch.from_numpy(eo), torch.from_numpy(ed), torch.rand(eo.shape[0], 1), 1 + torch.rand(eo.shape[0], 1)], -1)
    torch.manual_seed(11)
    jit = torch.rand(eo.shape[0], S)
    torch.manual_seed(11)
    z_ref = ref_renderer.NeRFRenderer(n_samples=S).sample_from_ray(rays)
    torch.manual_seed(11)
    z_ref2 = ref_utils.sample_from_rays_v2(rays, S)
    assert torch.equal(z_ref, z_ref2)

    # shell sampler
    torch.manual_seed(12)
    jit_shell = torch.rand(S)
    torch.manual_seed(12)
    xyz_sh, vd_sh, z_sh = ref_utils.sample_from_rays(ro, vd, 5.25, 9.75, S)
    xyz_fx, vd_fx, z_fx = ref_utils.sample_from_rays(ro, vd, 5.25, 9.75, S, z_fixed=True)

    # PE
    x = (torch.rand(50, 3) * 2 - 1) * 1.7
    pe10 = model_codenerf.PE(x, 10)
    pe4 = model_codenerf.PE(x, 4)

    # compositing: per-ray z, incl. opaque samples, negative sigmas, miss-ray style constant z
    N = 37
    sig = torch.randn(N, S) * 3
    sig[3] = 1e4  # opaque
    sig[4] = -1.0  # all empty
    rgbs = torch.rand(N, S, 3) * 1.5 - 0.25
    zv = torch.sort(torch.rand(N, S) * 4 + 2, -1)[0]
    zv[5] = 2.5  # miss ray: all samples at one point
    outs = {}
    for wb in (False, True):
        r = ref_renderer.NeRFRenderer(n_samples=S, white_bkgd=wb)
        s_, c_, z_ = sig.clone().requires_grad_(), rgbs.clone().requires_grad_(), zv.clone().requires_grad_()
        rgb, dep, acc = r.volume_render(s_, c_, z_)
        g = torch.Generator().manual_seed(5)
        g_rgb, g_dep, g_acc = torch.randn(N, 3, generator=g), torch.randn(N, generator=g), torch.randn(N, generator=g)
        (rgb * g_rgb).sum().add((dep * g_dep).sum()).add((acc * g_acc).sum()).backward()
        rgb3, dep3, acc3 = ref_renderer.volume_rendering3(sig.unsqueeze(-1), rgbs, zv, white_bkgd=wb)
        assert torch.equal(rgb3, rgb) and torch.equal(dep3, dep) and torch.equal(acc3, acc)
        outs.update({f"vr_rgb_wb{int(wb)}": rgb, f"vr_depth_wb{int(wb)}": dep, f"vr_acc_wb{int(wb)}": acc,
                     f"vr_gsig_wb{int(wb)}": s_.grad, f"vr_grgb_wb{int(wb)}": c_.grad, f"vr_gz_wb{int(wb)}": z_.grad,
                     "vr_up_rgb": g_rgb, "vr_up_depth": g_dep, "vr_up_acc": g_acc})
    # shared z (S,)
    z1 = zv[0].clone()
    rgb2, dep2, acc2 = ref_utils.volume_rendering2(sig.unsqueeze(-1), rgbs, z1)
    rgb1, dep1 = ref_utils.volume_rendering(torch.relu(sig).unsqueeze(-1), rgbs, z1)
    # batch (B,n,S) with z (B,S)
    Bb, nb = 3, 5
    sigb, rgbb, zb = sig[:Bb * nb].reshape(Bb, nb, S, 1), rgbs[:Bb * nb].reshape(Bb, nb, S, 3), zv[:Bb]
    rgbB, depB, accB = ref_utils.volume_rendering_batch(sigb, rgbb, zb)

    save("stages",
         K=K, c2w=c2w, roi=roi, rays_o=ro, viewdir=vd, rays_o_full=ro_full, viewdir_full=vd_full,
         x_vec=xv, y_vec=yv, rays_o_spec=ro_s, viewdir_spec=vd_s,
         box_o=eo, box_d=ed, box_half=half, box_hit_np=hit_np, box_zin_np=zi_np, box_zout_np=zo_np,
         box_hit_t=hit_t, box_zin_t=zi_t, box_zout_t=zo_t, box_hit_unit=hit_u, box_zin_unit=zi_u, box_zout_unit=zo_u,
         strat_rays=rays, strat_jitter=jit, strat_z=z_ref,
         shell_jitter=jit_shell, shell_xyz=xyz_sh, shell_z=z_sh, shell_z_fixed=z_fx,
         pe_x=x, pe10=pe10, pe4=pe4,
         vr_sig=sig, vr_rgbs=rgbs, vr_z=zv, vr2_rgb=rgb2, vr2_depth=dep2, vr2_acc=acc2, vr1_rgb=rgb1, vr1_depth=dep1,
         vrb_rgb=rgbB, vrb_depth=depB, vrb_acc=accB, **outs)


def golden_render_box():
    """Config-1 shape, scaled down: NeRFRenderer.render_rays (renderer.py:117) fwd + bwd, CodeNeRF()
    defaults, weights as shipped (requires_grad=True)."""
    seed, im_sz, S = 0, 12, 16
    sd = oracle.init_codenerf_state(seed=seed)
    torch.manual_seed(seed)
    model = model_codenerf.CodeNeRF()
    ref_sd = {k: v for k, v in model.state_dict().items()}
    assert all(torch.equal(ref_sd[k], sd[k]) for k in ref_sd), "oracle weight init != reference init"
    obj = oracle.synthetic_object(1, im_sz=im_sz)
    shp, tex = oracle.synthetic_latents(1, 1)
    cam = obj["cam_pose"].clone().requires_grad_()
    shp.requires_grad_(), tex.requires_grad_()
    r = ref_renderer.NeRFRenderer(n_samples=S)
    torch.manual_seed(100)
    jitter = torch.rand(im_sz * im_sz, S)
    torch.manual_seed(100)
    rgb, dep, acc, tgt, occ = r.render_rays(model, "cpu", obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"], obj["roi"],
                                            shp, tex, im_sz=im_sz)
    loss = losses(rgb, acc, tgt, occ)
    loss.backward()
    # hit mask straight from the reference's sampler on the same rays
    ro, vd = ref_utils.get_rays(obj["K"], obj["cam_pose"], obj["roi"], uv_steps=[im_sz, im_sz])
    torch.manual_seed(100)
    xyz, vdr, zv, hit = r.prepare_sampled_rays(ro, vd, obj["wlh"])
    g = {k: p.grad for k, p in model.named_parameters()}
    save("render_box_c1", sample=("gw_",),
         seed=seed, im_sz=im_sz, n_samples=S, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8),
         K=obj["K"], cam_pose=obj["cam_pose"], wlh=obj["wlh"], roi=obj["roi"], img=obj["img"], mask_occ=obj["mask_occ"],
         shapecode=shp, texturecode=tex, jitter=jitter,
         rgb=rgb, depth=dep, acc=acc, rgb_tgt=tgt, occ_pixels=occ, hit=hit, xyz=xyz, z_vals=zv, loss=loss,
         g_cam_pose=cam.grad, g_shapecode=shp.grad, g_texturecode=tex.grad,
         **{"gw_" + k: v for k, v in g.items()})


def golden_render_shell():
    """Config-3 shape, scaled down: utils.render_rays_v2 (utils.py:435) fwd + bwd with the SUPNeRF
    decoder (3/1/256), shapenet_obj_cood=1, the refine losses."""
    seed, im_sz, S = 2, 8, 16
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    model = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
    missing = model.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys
    obj = oracle.synthetic_object(5, im_sz=im_sz)
    shp, tex = oracle.synthetic_latents(5, 1)
    cam = obj["cam_pose"].clone().requires_grad_()
    shp.requires_grad_(), tex.requires_grad_()
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    torch.manual_seed(200)
    jitter = torch.rand(S)
    torch.manual_seed(200)
    rgb, dep, acc, tgt, occ = ref_utils.render_rays_v2(model, "cpu", obj["img"], obj["mask_occ"], cam, diag, obj["K"], obj["roi"],
                                                       S, shp, tex, 1, 0, im_sz=im_sz, n_rays=None)
    loss = losses(rgb, acc, tgt, occ)
    loss.backward()
    save("render_shell_c3",
         seed=seed, im_sz=im_sz, n_samples=S, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8),
         K=obj["K"], cam_pose=obj["cam_pose"], wlh=obj["wlh"], obj_diag=diag, roi=obj["roi"], img=obj["img"],
         mask_occ=obj["mask_occ"], shapecode=shp, texturecode=tex, jitter=jitter,
         rgb=rgb, depth=dep, acc=acc, rgb_tgt=tgt, occ_pixels=occ, loss=loss,
         g_cam_pose=cam.grad, g_shapecode=shp.grad, g_texturecode=tex.grad,
         gw_encoding_xyz_0_weight=model.encoding_xyz[0].weight.grad, gw_rgb_2_weight=model.rgb[2].weight.grad,
         gw_shape_latent_layer_2_0_weight=model.shape_latent_layer_2[0].weight.grad,
         gw_encoding_viewdir_0_weight=model.encoding_viewdir[0].weight.grad,
         gw_sigma_0_bias=model.sigma[0].bias.grad)


def golden_decoder_batch():
    """Config-2/5 shape, scaled down: AutoRFMix(3,1,256) decoder on B=2 objects, explicit xyz/viewdir
    (the trainer's call, trainer_unified_nuscenes.py:120-129), volume_rendering_batch, all grads."""
    seed, B, n, S = 3, 2, 24, 8
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    model = model_autorf.AutoRFMix(shape_blocks=3, texture_blocks=1, latent_dim=256)
    assert not model.load_state_dict(sd, strict=False).unexpected_keys
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(B, n, S, 3, generator=g) - 0.5).requires_grad_()
    vd = torch.nn.functional.normalize(torch.randn(B, n, 1, 3, generator=g), dim=-1).repeat(1, 1, S, 1).requires_grad_()
    zv = torch.sort(torch.rand(B, S, generator=g) * 4 + 6, -1)[0]
    shp, tex = oracle.synthetic_latents(seed, B)
    shp.requires_grad_(), tex.requires_grad_()
    sig, rgbs = model(xyz.flatten(0, 1), vd.flatten(0, 1), shp, tex)
    rgb, dep, acc = ref_utils.volume_rendering_batch(sig.reshape(B, n, S, 1), rgbs.reshape(B, n, S, 3), zv)
    tgt = torch.rand(B, n, 3, generator=g)
    occ = torch.sign(torch.randn(B, n, 1, generator=g))
    loss = losses(rgb, acc, tgt, occ)
    loss.backward()
    save("decoder_batch_c5", sample=("gw_",),
         seed=seed, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8),
         xyz=xyz, viewdir=vd, z_vals=zv, shapecode=shp, texturecode=tex, rgb_tgt=tgt, occ_pixels=occ,
         sigmas=sig, rgbs=rgbs, rgb=rgb, depth=dep, acc=acc, loss=loss,
         g_xyz=xyz.grad, g_viewdir=vd.grad, g_shapecode=shp.grad, g_texturecode=tex.grad,
         **{"gw_" + k: p.grad for k, p in model.named_parameters() if p.grad is not None})


def golden_autorf():
    """The non-mix AutoRF decoder (model_autorf.py:156-186), class defaults 5/5/128."""
    seed, B, n, S = 4, 2, 10, 6
    sd = oracle.init_autorf_state(seed=seed)
    model = model_autorf.AutoRF()
    assert not model.load_state_dict(sd, strict=False).unexpected_keys
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(B * n, S, 3, generator=g) - 0.5).requires_grad_()
    vd = torch.nn.functional.normalize(torch.randn(B * n, 1, 3, generator=g), dim=-1).repeat(1, S, 1).requires_grad_()
    shp, tex = oracle.synthetic_latents(seed, B, 128)
    shp.requires_grad_(), tex.requires_grad_()
    sig, rgbs = model(xyz, vd, shp, tex)
    up_s = torch.randn(sig.shape, generator=g)
    up_c = torch.randn(rgbs.shape, generator=g)
    ((sig * up_s).sum() + (rgbs * up_c).sum()).backward()
    save("autorf_decoder",
         seed=seed, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8),
         xyz=xyz, viewdir=vd, shapecode=shp, texturecode=tex, up_sigma=up_s, up_rgb=up_c, sigmas=sig, rgbs=rgbs,
         g_xyz=xyz.grad, g_viewdir=vd.grad, g_shapecode=shp.grad, g_texturecode=tex.grad,
         **{"gw_" + k: p.grad for k, p in model.named_parameters() if p.grad is not None and not k.startswith("img_encoder")})


def golden_scene_merge():
    """The merge step of the demo's scene compositor: the reference has no function for it, so the fixture EXECUTES the
    reference's own source lines (scripts/demo.py:560-569, read from the read-only tree, dedented) on synthetic samples of
    3 objects x 16 samples per ray, including rays that miss an object (z = -1, colour 1, sigma 0: demo.py:541, 555-556)."""
    import textwrap
    src = open("/root/reference/scripts/demo.py").read().splitlines()
    block = textwrap.dedent("\n".join(src[559:569]))        # lines 560-569 (1-based)
    assert block.lstrip().startswith("# sort by z values") and "z_args = torch.searchsorted(z_sort, z_vals)" in block and \
        block.rstrip().endswith("volume_rendering3(sigmas_sort, rgbs_sort, z_sort, white_bkgd=True)"), block
    g = torch.Generator().manual_seed(12)
    Nr, Nb, n_samples = 64, 3, 16
    z = torch.rand(Nr * Nb, n_samples, generator=g).sort(-1).values * 6 + 4 + torch.rand(Nr * Nb, 1, generator=g) * 3
    sig = torch.rand(Nr * Nb, n_samples, generator=g) * 3 - 0.5
    rgb = torch.rand(Nr * Nb, n_samples, 3, generator=g)
    empty = torch.rand(Nr * Nb, 1, generator=g) < 0.3                     # this object is missed by this ray
    z = torch.where(empty, torch.full_like(z, -1.0), z)
    z[5, 3] = z[5, 7]                                                      # a genuine tie between two samples
    sig = torch.where(empty, torch.zeros_like(sig), sig)
    rgb = torch.where(empty.unsqueeze(-1), torch.ones_like(rgb), rgb)
    env = dict(z_vals=z.clone(), sigmas=sig.clone(), rgbs=rgb.clone(), Nb=Nb, n_samples=n_samples, torch=torch,
               volume_rendering3=ref_renderer.volume_rendering3)
    exec(block, env)
    save("scene_merge", n_objects=np.int64(Nb), n_samples=np.int64(n_samples), z_vals=z.view(-1, Nb * n_samples),
         sigmas=sig.view(-1, Nb * n_samples), rgbs=rgb.view(-1, Nb * n_samples, 3), z_sort=env["z_sort"], z_args=env["z_args"],
         sigmas_sort=env["sigmas_sort"], rgbs_sort=env["rgbs_sort"], rgb=env["rgb"], depth=env["depth"], acc=env["weights"])


def golden_drivers():
    """The remaining public drivers of SURVEY 8(b), each executed through the UNMODIFIED reference on one small object:
    renderer.render_rays_v3 (full grid and a random ray subset), utils.render_rays / render_rays_specified /
    prepare_pixel_samples / render_full_img, NeRFRenderer.render_rays_specified / prepare_pixel_samples / render_full_img.
    Every torch.rand_like draw of the box stack is recorded (the CUDA path draws on the device generator: the tests feed the
    recorded jitter back); the shell stack draws torch.rand(S) on the CPU generator on both sides (same seed, same numbers)."""
    seed, S_box, S = 7, 64, 16
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    model = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
    assert not model.load_state_dict(sd, strict=False).unexpected_keys
    model.requires_grad_(False)
    obj = oracle.synthetic_object(seed, im_sz=8)
    shp0, tex0 = oracle.synthetic_latents(seed, 1)
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    # a small full-resolution crop (12 x 10 pixels) around the projected box centre, with its own image / coherent +-1 mask
    r = [int(v) for v in obj["roi"]]
    cx, cy = (r[0] + r[2]) // 2, (r[1] + r[3]) // 2
    roi_s = torch.tensor([cx - 6, cy - 5, cx + 6, cy + 5], dtype=torch.int32)
    g = torch.Generator().manual_seed(seed)
    img_s = torch.rand(10, 12, 3, generator=g)
    mask_s = torch.ones(10, 12, 1)
    mask_s[:, 7:] = -1.0
    mask_s[:2] = 0.0
    x_vec = np.array([0, 3, 11, 5, 7, 2, 9], dtype=np.int64)
    y_vec = np.array([0, 9, 4, 5, 1, 8, 3], dtype=np.int64)
    out = dict(seed=seed, wlh=obj["wlh"], obj_diag=diag, K=obj["K"], cam_pose=obj["cam_pose"], roi=obj["roi"], img=obj["img"],
               mask_occ=obj["mask_occ"], roi_s=roi_s, img_s=img_s, mask_s=mask_s, x_vec=x_vec, y_vec=y_vec, shapecode=shp0,
               texturecode=tex0, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8))

    draws = []
    orig_rand_like = torch.rand_like

    def recording_rand_like(t, *a, **k):
        v = orig_rand_like(t, *a, **k)
        draws.append(v.clone())
        return v

    def leaves():
        return obj["cam_pose"].clone().requires_grad_(), shp0.clone().requires_grad_(), tex0.clone().requires_grad_()

    torch.rand_like = recording_rand_like
    try:
        # ---- renderer.render_rays_v3 (renderer.py:382): full 8x8 grid, shapenet frame, adjust_scale, fwd + bwd
        cam, shp, tex = leaves()
        torch.manual_seed(70)
        rgb, dep, acc, tgt, occ = ref_renderer.render_rays_v3(model, "cpu", obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"], obj["roi"],
                                                             S_box, shp, tex, 1, 0, im_sz=8, n_rays=None, adjust_scale=1.1)
        loss = losses(rgb, acc, tgt, occ)
        loss.backward()
        out.update(v3_jitter=draws.pop(), v3_rgb=rgb, v3_depth=dep, v3_acc=acc, v3_tgt=tgt, v3_occ=occ, v3_loss=loss,
                   v3_g_cam=cam.grad, v3_g_shp=shp.grad, v3_g_tex=tex.grad)
        assert not draws
        # ---- ... with a random ray subset (np.random.permutation under a fixed numpy seed)
        cam, shp, tex = leaves()
        np.random.seed(71)
        torch.manual_seed(71)
        rgb, dep, acc, tgt, occ = ref_renderer.render_rays_v3(model, "cpu", obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"], obj["roi"],
                                                             S_box, shp, tex, 0, 0, im_sz=8, n_rays=20)
        out.update(v3s_jitter=draws.pop(), v3s_rgb=rgb, v3s_depth=dep, v3s_acc=acc, v3s_tgt=tgt, v3s_occ=occ)
        # ---- NeRFRenderer drivers on the small full-resolution crop
        R = ref_renderer.NeRFRenderer(n_samples=S)
        cam, shp, tex = leaves()
        torch.manual_seed(72)
        rgb, dep, acc, tgt, occ = R.render_rays_specified(model, "cpu", img_s, mask_s, cam, obj["wlh"], obj["K"], roi_s, x_vec, y_vec, shp, tex)
        loss = losses(rgb, acc, tgt, occ)
        loss.backward()
        out.update(rs_jitter=draws.pop(), rs_rgb=rgb, rs_depth=dep, rs_acc=acc, rs_tgt=tgt, rs_occ=occ, rs_g_cam=cam.grad,
                   rs_g_shp=shp.grad, rs_g_tex=tex.grad)
        np.random.seed(73)
        torch.manual_seed(73)
        xyz, vd, zv, tgt, occ = R.prepare_pixel_samples(img_s, mask_s, obj["cam_pose"], obj["wlh"], obj["K"], roi_s, 40)
        out.update(rp_jitter=draws.pop(), rp_xyz=xyz, rp_viewdir=vd, rp_z_vals=zv, rp_tgt=tgt, rp_occ=occ)
        torch.manual_seed(74)
        with torch.no_grad():
            im_full, dep_full = R.render_full_img(model, "cpu", obj["cam_pose"], obj["wlh"], obj["K"], roi_s, shp0, tex0, out_depth=True)
        out.update(rf_jitter=draws.pop(), rf_img=im_full, rf_depth=dep_full)
        # ---- the kitti2nusc frame rotation (renderer.py:153-163; no shipped caller enables it) through NeRFRenderer.render_rays
        R64 = ref_renderer.NeRFRenderer(n_samples=S)
        cam, shp, tex = leaves()
        torch.manual_seed(79)
        rgb, dep, acc, tgt, occ = R64.render_rays(model, "cpu", obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"], obj["roi"], shp, tex,
                                                  kitti2nusc=True, im_sz=8)
        loss = losses(rgb, acc, tgt, occ)
        loss.backward()
        out.update(k2n_jitter=draws.pop(), k2n_rgb=rgb, k2n_depth=dep, k2n_acc=acc, k2n_tgt=tgt, k2n_occ=occ, k2n_g_cam=cam.grad,
                   k2n_g_shp=shp.grad, k2n_g_tex=tex.grad)
        assert not draws
    finally:
        torch.rand_like = orig_rand_like
    # ---- utils.render_rays_v2 with the symmetric augmentation taken (python `random`: seed 2 draws 0.956 > 0.5) and kitti2nusc
    import random as _random
    cam, shp, tex = leaves()
    _random.seed(2)
    torch.manual_seed(80)
    rgb, dep, acc, tgt, occ = ref_utils.render_rays_v2(model, "cpu", obj["img"], obj["mask_occ"], cam, diag, obj["K"], obj["roi"], S, shp, tex,
                                                       1, 1, kitti2nusc=True, im_sz=8, n_rays=None)
    loss = losses(rgb, acc, tgt, occ)
    loss.backward()
    out.update(sym_rgb=rgb, sym_depth=dep, sym_acc=acc, sym_tgt=tgt, sym_occ=occ, sym_g_cam=cam.grad, sym_g_shp=shp.grad, sym_g_tex=tex.grad)
    # ---- utils drivers (shell stack: one torch.rand(S) on the CPU generator per call)
    cam, shp, tex = leaves()
    np.random.seed(75)
    torch.manual_seed(75)
    rgb, dep, acc, tgt, occ = ref_utils.render_rays(model, "cpu", img_s, mask_s, cam, diag, obj["K"], roi_s, S, shp, tex, 1, 0, n_rays=50)
    loss = losses(rgb, acc, tgt, occ)
    loss.backward()
    out.update(ur_rgb=rgb, ur_depth=dep, ur_acc=acc, ur_tgt=tgt, ur_occ=occ, ur_g_cam=cam.grad, ur_g_shp=shp.grad, ur_g_tex=tex.grad)
    cam, shp, tex = leaves()
    torch.manual_seed(76)
    rgb, dep, acc, tgt, occ = ref_utils.render_rays_specified(model, "cpu", img_s, mask_s, cam, diag, obj["K"], roi_s, x_vec, y_vec, S, shp, tex, 1, 0)
    out.update(us_rgb=rgb, us_depth=dep, us_acc=acc, us_tgt=tgt, us_occ=occ)
    np.random.seed(77)
    torch.manual_seed(77)
    xyz, vd, zv, tgt, occ = ref_utils.prepare_pixel_samples(img_s, mask_s, obj["cam_pose"], diag, obj["K"], roi_s, 40, S, 1, 0)
    out.update(up_xyz=xyz, up_viewdir=vd, up_z_vals=zv, up_tgt=tgt, up_occ=occ)
    torch.manual_seed(78)
    with torch.no_grad():
        im_full, dep_full = ref_utils.render_full_img(model, "cpu", obj["cam_pose"], obj["wlh"], obj["K"], roi_s, S, shp0, tex0, 1, out_depth=True)
    out.update(uf_img=im_full, uf_depth=dep_full)
    save("drivers", **out)


def golden_drivers_truth64():
    """fp64 TRUTH for the driver gradients of tests/golden/drivers.npz: the same UNMODIFIED reference drivers executed with
    torch's default dtype set to float64 (model.double(), float64 inputs, the fp32 fixture's recorded jitter replayed), so that the
    GPU tests can tell a kernel's error from the fp32 reference's own (pose gradients are sums with heavy cancellation: the
    reference's fp32 value is 3e-3 .. 5e-3 away from this truth, its latent gradients up to 4e-5).  Host-side float32 roundings
    the reference makes explicitly (`.astype(np.float32)`, renderer.py:92,97-100) are part of its semantics and stay."""
    import random as _random
    g = dict(np.load(os.path.join(OUT, "drivers.npz")))
    seed = int(g["seed"])
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    orig_rand_like = torch.rand_like
    orig_from_numpy = torch.from_numpy
    try:
        # the kitti2nusc rotation is built as a float32 numpy matrix of 0 / +-1 entries (renderer.py:154-157, utils.py:481-484) and
        # `@` does not promote: hand float32 arrays over as float64 (same values) for this run only
        torch.from_numpy = lambda a: orig_from_numpy(a).double() if a.dtype == np.float32 else orig_from_numpy(a)
        model = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
        model.load_state_dict(sd, strict=False)
        model = model.double()
        model.requires_grad_(False)
        T_ = lambda a: orig_from_numpy(np.asarray(a))   # noqa: E731
        D_ = lambda a: T_(a).double()                     # noqa: E731

        def leaves():
            return D_(g["cam_pose"]).requires_grad_(), D_(g["shapecode"]).requires_grad_(), D_(g["texturecode"]).requires_grad_()

        def replay(key):
            torch.rand_like = lambda t, *a, **k: D_(g[key])

        out = {}

        def finish(pre, res, cam, shp, tex):
            rgb, dep, acc, tgt, occ = res
            losses(rgb, acc, tgt, occ).backward()
            for name, t32 in (("rgb", rgb), ("depth", dep), ("acc", acc)):   # same render as the fp32 fixture (no flipped hit masks)
                e = float((t32.detach() - D_(g[pre + "_" + name])).abs().max() / D_(g[pre + "_" + name]).abs().max())
                assert e < 2e-5, (pre, name, e)
            out.update({pre + "_g_cam64": cam.grad, pre + "_g_shp64": shp.grad, pre + "_g_tex64": tex.grad})

        img, mask, K, roi, wlh = D_(g["img"]), D_(g["mask_occ"]), D_(g["K"]), T_(g["roi"]), g["wlh"]
        img_s, mask_s, roi_s, diag = D_(g["img_s"]), D_(g["mask_s"]), T_(g["roi_s"]), np.float32(g["obj_diag"])
        cam, shp, tex = leaves()
        replay("v3_jitter")
        finish("v3", ref_renderer.render_rays_v3(model, "cpu", img, mask, cam, wlh, K, roi, 64, shp, tex, 1, 0, im_sz=8, n_rays=None,
                                                 adjust_scale=1.1), cam, shp, tex)
        R = ref_renderer.NeRFRenderer(n_samples=16)
        cam, shp, tex = leaves()
        replay("rs_jitter")
        finish("rs", R.render_rays_specified(model, "cpu", img_s, mask_s, cam, wlh, K, roi_s, g["x_vec"], g["y_vec"], shp, tex), cam, shp, tex)
        cam, shp, tex = leaves()
        replay("k2n_jitter")
        finish("k2n", R.render_rays(model, "cpu", img, mask, cam, wlh, K, roi, shp, tex, kitti2nusc=True, im_sz=8), cam, shp, tex)
        torch.rand_like = orig_rand_like
        # shell stack: torch.rand(S) on the CPU generator; drawn in float32 under the fixture's seed (the generator's float64 stream
        # differs), then handed to the float64 run
        def shell_rand(seed_):
            torch.manual_seed(seed_)
            j = torch.rand(16, dtype=torch.float32).double()
            orig = torch.rand
            torch.rand = lambda *a, **k: j
            return orig
        cam, shp, tex = leaves()
        _random.seed(2)
        orig = shell_rand(80)
        try:
            res = ref_utils.render_rays_v2(model, "cpu", img, mask, cam, diag, K, roi, 16, shp, tex, 1, 1, kitti2nusc=True, im_sz=8, n_rays=None)
        finally:
            torch.rand = orig
        finish("sym", res, cam, shp, tex)
        cam, shp, tex = leaves()
        np.random.seed(75)
        orig = shell_rand(75)
        try:
            res = ref_utils.render_rays(model, "cpu", img_s, mask_s, cam, diag, K, roi_s, 16, shp, tex, 1, 0, n_rays=50)
        finally:
            torch.rand = orig
        finish("ur", res, cam, shp, tex)
    finally:
        torch.rand_like = orig_rand_like
        torch.from_numpy = orig_from_numpy
        torch.set_default_dtype(old)
    save("drivers_truth64", **out)


def golden_pose_estimator():
    """SURVEY 8f rank 2 through the UNMODIFIED reference: SUPNeRF.encode_img (eval and train mode batch norm) + pose_update
    (model_supnerf.py:108-152, 218-239), the box-corner projection helpers (utils.py:1032-1147, 1175-1197) and one whole
    ParallelModel.forward of the joint trainer (trainer_unified_nuscenes.py:27-148) with its backward.  The trainer imports
    pytorch3d's axis-angle maps, which are not part of the reference tree (SURVEY 8c): they are stubbed with the package's Rodrigues
    restatement, so everything except those two maps is the reference's own arithmetic.  Weights: synthetic.pose_estimator_state."""
    from supnerf_b200 import pose_estimator as pe, synthetic
    seed = 21
    model = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
    sd = dict(oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed))
    sd.update(synthetic.pose_estimator_state(model.state_dict(), seed))
    assert set(sd) == set(model.state_dict())
    model.load_state_dict(sd)
    g = torch.Generator().manual_seed(seed)
    B = 2
    img = torch.rand(B, 3, 128, 128, generator=g)
    out = dict(seed=seed, img=img, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8))
    model.eval()
    img_r = img.clone().requires_grad_()
    f_s, f_t, f_p, uv, _ = model.encode_img(img_r)
    uv_src = torch.rand(B, 16, generator=g) * 2 - 1
    delta = model.pose_update(f_p, uv_src)
    up = [torch.randn(t.shape, generator=g) for t in (f_s, f_t, f_p, uv, delta)]
    model.zero_grad()
    sum((t * u).sum() for t, u in zip((f_s, f_t, f_p, uv, delta), up)).backward()
    out.update(eval_shape=f_s, eval_texture=f_t, eval_pose=f_p, eval_uv=uv, uv_src=uv_src, eval_delta=delta,
               up_shape=up[0], up_texture=up[1], up_pose=up[2], up_uv=up[3], up_delta=up[4], eval_g_img=img_r.grad,
               eval_gw_conv1=model.img_encoder.conv1.weight.grad, eval_gw_fc_pose=model.img_encoder.fc_pose.weight.grad,
               eval_gw_l4pose_conv=model.img_encoder.layer4_pose[2].conv2.weight.grad[::16, ::16].contiguous(),   # a strided slice: small fixture
               
               eval_gw_out_delta=model.out_delta_layer.weight.grad, eval_gw_regress0=model.regress_layer_0[0].weight.grad)
    model.train()
    with torch.no_grad():
        f_s, f_t, f_p, uv, _ = model.encode_img(img)
    out.update(train_shape=f_s, train_texture=f_t, train_pose=f_p, train_uv=uv,
               train_running_mean_bn1=model.img_encoder.bn1.running_mean.clone())
    # ---- box-corner projection helpers
    objs = [oracle.synthetic_object(seed + i, im_sz=16) for i in range(B)]
    c2o = torch.stack([o["cam_pose"] for o in objs])                       # camera -> object
    R_o2c = c2o[:, :, :3].transpose(1, 2)
    obj_pose = torch.cat([R_o2c, -R_o2c @ c2o[:, :, 3:]], -1).contiguous()  # object -> camera (the trainer's obj_poses)
    wlh = torch.stack([torch.from_numpy(np.asarray(o["wlh"], dtype=np.float32)) for o in objs])
    K = torch.stack([o["K"] for o in objs])
    roi = torch.stack([torch.as_tensor(np.asarray(o["roi"]), dtype=torch.float32) for o in objs])
    corners = ref_utils.corners_of_box_batch(obj_pose, wlh)
    corners_k = ref_utils.corners_of_box_batch(obj_pose, wlh, is_kitti=True, scale=1.1)
    uv_all = ref_utils.view_points_batch(corners, K, normalize=True)
    uv_norm, dim = ref_utils.normalize_by_roi(uv_all[:, :2, :], roi, need_square=True)
    uv_norm2, _ = ref_utils.normalize_by_roi(uv_all[:, :2, :], roi, need_square=False)
    out.update(obj_pose=obj_pose, wlh=wlh, K=K, roi=roi, corners=corners, corners_kitti=corners_k, uv_all=uv_all, uv_norm=uv_norm,
               uv_dim=dim, uv_norm_nonsquare=uv_norm2)
    # ---- one joint training step (ParallelModel.forward + backward), pytorch3d's two maps stubbed
    stubs = {}
    for name in ("wandb", "torch.utils.tensorboard", "pytorch3d", "pytorch3d.transforms", "pytorch3d.transforms.rotation_conversions",
                 "imageio", "skimage", "skimage.metrics"):
        if name not in sys.modules:
            stubs[name] = sys.modules[name] = types.ModuleType(name)
    sys.modules["torch.utils.tensorboard"].SummaryWriter = object
    rc = sys.modules["pytorch3d.transforms.rotation_conversions"]
    rc.matrix_to_axis_angle, rc.axis_angle_to_matrix = pe.matrix_to_axis_angle_batch, pe.axis_angle_to_matrix_batch
    sys.modules["pytorch3d.transforms"].rotation_conversions = rc
    sys.modules["pytorch3d"].transforms = sys.modules["pytorch3d.transforms"]
    if "skimage.metrics" in stubs:
        sys.modules["skimage.metrics"].structural_similarity = None
    import trainer_unified_nuscenes as tun
    hp = {"loss_pose_coef": 0.01, "loss_code_coef": 0.1, "loss_occ_coef": 0.1}
    pm = tun.ParallelModel(model, hp, im_enc_rate=1.0, pred_wlh=False)
    n, S_ = 48, 16
    xyz = (torch.rand(B, n, S_, 3, generator=g) - 0.5) * 1.2
    vd = torch.nn.functional.normalize(torch.randn(B, n, 1, 3, generator=g), dim=-1).repeat(1, 1, S_, 1)
    zv = (torch.rand(B, S_, generator=g).sort(-1).values * 4 + 8)   # one shared sample vector per object (the shell stack)
    tgt = torch.rand(B, n, 3, generator=g)
    occ = torch.randint(-1, 2, (B, n, 1), generator=g).float()
    shp, tex = oracle.synthetic_latents(seed, B)
    shp, tex = shp.clone().requires_grad_(), tex.clone().requires_grad_()
    # a perturbed source pose: small rotation about z + a translation error
    ang = torch.tensor([0.15, -0.1])
    Rz = torch.stack([torch.stack([torch.stack([torch.cos(a), -torch.sin(a), torch.zeros(())]), torch.stack([torch.sin(a), torch.cos(a), torch.zeros(())]),
                                   torch.tensor([0., 0., 1.])]) for a in ang])
    src_pose = torch.cat([obj_pose[:, :, :3] @ Rz, obj_pose[:, :, 3:] * torch.tensor([1.03, 0.98, 1.05]).view(1, 3, 1)], -1)
    tgt_uv = uv_all[:, :2, :]
    model.train()
    model.zero_grad()
    import random as _random
    _random.seed(0)   # enc_active = random.uniform(0, 1) < 1.0: always taken
    losses_all, loss_total, shp_out, tex_out, pred_pose3, pred_uv_direct = pm(img, shp, tex, xyz, vd, zv, tgt, occ, src_pose, tgt_uv, wlh, roi, K,
                                                                              wlh, tgt_uv)
    loss_total.mean().backward()
    out.update(j_xyz=xyz, j_viewdir=vd, j_z_vals=zv, j_rgb_tgt=tgt, j_occ=occ, j_shapecode=shp.detach(), j_texturecode=tex.detach(),
               j_src_pose=src_pose, j_tgt_uv=tgt_uv, j_loss_total=loss_total.detach(), j_shapecode_out=shp_out, j_texturecode_out=tex_out,
               j_pred_pose3=pred_pose3, j_pred_uv_direct=pred_uv_direct, j_g_shapecode=shp.grad, j_g_texturecode=tex.grad,
               j_gw_conv1=model.img_encoder.conv1.weight.grad, j_gw_fc_shape=model.img_encoder.fc_shape.weight.grad,
               j_gw_out_delta=model.out_delta_layer.weight.grad, j_gw_encoding_xyz=model.encoding_xyz[0].weight.grad,
               j_gw_rgb2=model.rgb[2].weight.grad)
    for k_, v_ in losses_all.items():
        if k_ != "psnr":
            out["j_" + k_] = v_.detach() if torch.is_tensor(v_) else torch.tensor(v_)
    # ---- the same joint step in float64 (default dtype float64, model.double(), float32 numpy constants handed over as float64):
    # the TRUTH for its gradients (sums over all samples with cancellation: see conftest.parity)
    old_dt = torch.get_default_dtype()
    orig_from_numpy = torch.from_numpy
    torch.set_default_dtype(torch.float64)
    torch.from_numpy = lambda a: orig_from_numpy(a).double() if a.dtype == np.float32 else orig_from_numpy(a)
    try:
        model64 = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
        model64.load_state_dict(sd)
        model64 = model64.double()
        model64.train()
        pm64 = tun.ParallelModel(model64, hp, im_enc_rate=1.0, pred_wlh=False)
        shp64, tex64 = shp.detach().double().requires_grad_(), tex.detach().double().requires_grad_()
        D_ = lambda t: t.detach().double()   # noqa: E731
        _random.seed(0)
        _, total64, *_ = pm64(D_(img), shp64, tex64, D_(xyz), D_(vd), D_(zv), D_(tgt), D_(occ), D_(src_pose), D_(tgt_uv), D_(wlh), D_(roi), D_(K),
                              D_(wlh), D_(tgt_uv))
        total64.mean().backward()
        e64 = model64.img_encoder
        out.update(j64_loss_total=total64.detach(), j64_g_shapecode=shp64.grad, j64_g_texturecode=tex64.grad,
                   j64_gw_conv1=e64.conv1.weight.grad, j64_gw_fc_shape=e64.fc_shape.weight.grad, j64_gw_out_delta=model64.out_delta_layer.weight.grad,
                   j64_gw_encoding_xyz=model64.encoding_xyz[0].weight.grad, j64_gw_rgb2=model64.rgb[2].weight.grad)
    finally:
        torch.from_numpy = orig_from_numpy
        torch.set_default_dtype(old_dt)
    for name in stubs:
        sys.modules.pop(name, None)
    save("pose_estimator", sample=("eval_g", "j_gw_", "j64_gw_"), **out)


def golden_scene():
    """The whole scene compositor of the demo (SURVEY 8f rank 4): the reference's `vis_scene` method (scripts/demo.py:425-579) is
    EXECUTED as it stands (its source text is read from the read-only tree and exec-ed; `self` is a plain namespace carrying the
    attributes it reads) on three synthetic cars in a 64 x 48 image, box-bounded rays, 16 samples, several ray batches.  Every
    torch.rand_like draw is recorded (the reference draws on the CPU generator)."""
    import textwrap
    import tqdm
    src = open("/root/reference/scripts/demo.py").read().splitlines()
    start = next(i for i, l in enumerate(src) if l.startswith("    def vis_scene("))
    end = next(i for i in range(start, len(src)) if src[i].strip() == "return canvas")
    fn_src = textwrap.dedent("\n".join(src[start:end + 1]))
    env = dict(torch=torch, np=np, tqdm=tqdm, corners_of_box_batch=ref_utils.corners_of_box_batch, view_points_batch=ref_utils.view_points_batch,
               roi_process=ref_utils.roi_process, get_rays=ref_utils.get_rays, ray_box_intersection=ref_utils.ray_box_intersection,
               sample_from_rays_v2=ref_utils.sample_from_rays_v2, volume_rendering3=ref_renderer.volume_rendering3)
    exec(fn_src, env)
    seed, Nb, H, W, S = 33, 3, 48, 64, 16
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    model = model_supnerf.SUPNeRF(shape_blocks=3, texture_blocks=1, pose_blocks=3, regress_blocks=3, latent_dim=256)
    model.load_state_dict(sd, strict=False)
    model.requires_grad_(False)
    g = torch.Generator().manual_seed(seed)
    base = torch.tensor([[0., -1., 0.], [0., 0., -1.], [1., 0., 0.]])
    poses = []
    for yaw, t in ((0.4, (-2.2, 0.3, 9.0)), (-1.1, (1.5, 0.2, 11.0)), (2.0, (0.2, 0.4, 14.0))):
        Rz = torch.tensor([[np.cos(yaw), -np.sin(yaw), 0.], [np.sin(yaw), np.cos(yaw), 0.], [0., 0., 1.]], dtype=torch.float32)
        poses.append(torch.cat([base @ Rz, torch.tensor(t).view(3, 1)], 1))
    obj_poses = torch.stack(poses)
    obj_wlh = torch.tensor([[1.9, 4.6, 1.7], [2.0, 4.9, 1.6], [1.8, 4.3, 1.8]])
    K = torch.tensor([[60., 0., 32.], [0., 60., 24.], [0., 0., 1.]])
    shp, tex = oracle.synthetic_latents(seed, Nb)
    me = types.SimpleNamespace(obj_poses=obj_poses, obj_wlh=obj_wlh, hpams={"dataset": {"img_h": H, "img_w": W}, "n_samples": S, "shapenet_obj_cood": 1},
                               rend_aabb=True, ray_batch_size=300, adjust_scale=1.1, model=model, device="cpu", shapecodes=shp, texturecodes=tex)
    draws = []
    orig = torch.rand_like

    def rec(t, *a, **k):
        v = orig(t, *a, **k)
        draws.append(v.clone())
        return v
    torch.rand_like = rec
    try:
        torch.manual_seed(seed)
        canvas = env["vis_scene"](me, {"cam_intrinsics": K}, [0.3, -0.1, 1.0])
    finally:
        torch.rand_like = orig
    jitter = torch.cat(draws, 0).view(-1, Nb, S)
    save("scene", seed=seed, H=H, W=W, n_samples=S, K=K, obj_poses=obj_poses, obj_wlh=obj_wlh, shapecodes=shp, texturecodes=tex,
         manipulation=np.asarray([0.3, -0.1, 1.0], dtype=np.float32), adjust_scale=np.float32(1.1), ray_batch_size=np.int64(300), jitter=jitter,
         canvas=canvas, weights_sha256=np.frombuffer(state_hash(sd).encode(), dtype=np.uint8))
    print("scene: valid rays", jitter.shape[0], "non-white pixels", int((canvas != 255).any(-1).sum()))


def golden_state_dict_keys():
    """state_dict key -> shape of the reference modules (the checkpoint ABI, SURVEY 8b): lets the CPU tests check that the
    drop-in modules load a reference checkpoint with the default strict=True without importing the reference."""
    import json
    out = {}
    for name, mod in (("CodeNeRF", model_codenerf.CodeNeRF()), ("AutoRFMix_3_1_256", model_autorf.AutoRFMix(3, 1, 256)),
                      ("AutoRF", model_autorf.AutoRF()), ("SUPNeRF_3_1_3_3_256", model_supnerf.SUPNeRF(3, 1, 3, 3, 256))):
        out[name] = {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in mod.state_dict().items()}
    path = os.path.join(OUT, "state_dict_keys.json")
    json.dump(out, open(path, "w"))
    print("wrote", path, {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    torch.set_num_threads(8)
    golden_stages()
    golden_render_box()
    golden_render_shell()
    golden_decoder_batch()
    golden_autorf()
    golden_scene_merge()
    golden_drivers()
    golden_drivers_truth64()
    golden_pose_estimator()
    golden_scene()
    golden_state_dict_keys()
