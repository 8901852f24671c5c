"""Pins oracle/oracle.py against fixtures produced by the unmodified reference (tools/make_golden.py).
The weight gradients of render_box_c1 and decoder_batch_c5 are stored as a strided sample of 1/2 .. 1/9 of their elements
(conftest.Sampled): they are judged on those elements, against max|.| of the whole array."""
import hashlib

import numpy as np
import torch

from conftest import T, load_golden, rel_err
from oracle import oracle

TOL = 2e-6  # fp32 restatement vs fp32 reference on the same CPU: op order is identical up to reductions


def _hash(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def _check_weights(g, sd):
    assert _hash(sd) == bytes(g["weights_sha256"]).decode(), "seeded weight init drifted from the fixture"


def test_rays_bit_exact():
    g = load_golden("stages")
    ro, vd = oracle.get_rays(T(g["K"]), T(g["c2w"]), g["roi"], uv_steps=[12, 12])
    assert torch.equal(ro, T(g["rays_o"])) and torch.equal(vd, T(g["viewdir"]))
    ro, vd = oracle.get_rays(T(g["K"]), T(g["c2w"]), [100, 50, 109, 57])
    assert torch.equal(ro, T(g["rays_o_full"])) and torch.equal(vd, T(g["viewdir_full"]))
    ro, vd = oracle.get_rays_specified(T(g["K"]), T(g["c2w"]), g["x_vec"] + g["roi"][0], g["y_vec"] + g["roi"][1])
    assert torch.equal(ro, T(g["rays_o_spec"])) and torch.equal(vd, T(g["viewdir_spec"]))


def test_slab_hit_mask_bit_exact():
    g = load_golden("stages")
    o, d, half = g["box_o"], g["box_d"], g["box_half"]
    n = o.shape[0]
    amin, amax = np.repeat(-half[None], n, 0), np.repeat(half[None], n, 0)
    tn, tf, hit = oracle.ray_box_intersection_np(o, d, amin, amax)
    assert np.array_equal(hit, g["box_hit_np"])
    assert np.array_equal(tn[hit], g["box_zin_np"]) and np.array_equal(tf[hit], g["box_zout_np"])
    tn, tf, hit = oracle.ray_box_intersection(T(o), T(d), T(amin), T(amax))
    assert np.array_equal(hit.numpy(), g["box_hit_t"])
    assert np.array_equal(tn[hit].numpy(), g["box_zin_t"]) and np.array_equal(tf[hit].numpy(), g["box_zout_t"])
    tn, tf, hit = oracle.ray_box_intersection(T(o), T(d), -torch.ones(n, 3), torch.ones(n, 3))
    assert np.array_equal(hit.numpy(), g["box_hit_unit"]) and np.array_equal(tn[hit].numpy(), g["box_zin_unit"])
    assert hit.any() and not hit.all()


def test_stratified_and_shell_bit_exact():
    g = load_golden("stages")
    rays = T(g["strat_rays"])
    z = oracle.stratified_z(rays[:, 6:7], rays[:, 7:8], 16, T(g["strat_jitter"]))
    assert torch.equal(z, T(g["strat_z"]))
    k = torch.floor((z - rays[:, 6:7]) / (rays[:, 7:8] - rays[:, 6:7]) * 16).long()
    assert ((k - torch.arange(16)[None]).abs() <= 0).float().mean() > 0.99  # stratum index of every sample
    xyz, vd, zs = oracle.sample_from_rays_shell(T(g["rays_o"]), T(g["viewdir"]), 5.25, 9.75, 16, T(g["shell_jitter"]))
    assert torch.equal(zs, T(g["shell_z"])) and torch.equal(xyz, T(g["shell_xyz"]))
    _, _, zf = oracle.sample_from_rays_shell(T(g["rays_o"]), T(g["viewdir"]), 5.25, 9.75, 16, None)
    assert torch.equal(zf, T(g["shell_z_fixed"]))


def test_pe_bit_exact():
    g = load_golden("stages")
    assert torch.equal(oracle.positional_encoding(T(g["pe_x"]), 10), T(g["pe10"]))
    assert torch.equal(oracle.positional_encoding(T(g["pe_x"]), 4), T(g["pe4"]))


def test_composite_variants():
    g = load_golden("stages")
    sig, rgbs, z = T(g["vr_sig"]), T(g["vr_rgbs"]), T(g["vr_z"])
    for wb in (0, 1):
        s_, c_, z_ = sig.clone().requires_grad_(), rgbs.clone().requires_grad_(), z.clone().requires_grad_()
        rgb, dep, acc = oracle.composite(s_, c_, z_, bool(wb))
        assert torch.equal(rgb, T(g[f"vr_rgb_wb{wb}"])) and torch.equal(dep, T(g[f"vr_depth_wb{wb}"]))
        assert torch.equal(acc, T(g[f"vr_acc_wb{wb}"]))
        up = T(g["vr_up_rgb"]), T(g["vr_up_depth"]), T(g["vr_up_acc"])
        ((rgb * up[0]).sum() + (dep * up[1]).sum() + (acc * up[2]).sum()).backward()
        assert rel_err(s_.grad, g[f"vr_gsig_wb{wb}"]) < TOL and rel_err(c_.grad, g[f"vr_grgb_wb{wb}"]) < TOL
        assert rel_err(z_.grad, g[f"vr_gz_wb{wb}"]) < TOL
        # closed form (the K3b spec) against the reference's autograd, in fp64 to separate formula from rounding
        gs, gc, gz = oracle.composite_backward_closed_form(sig.double(), rgbs.double(), z.double(), up[0].double(),
                                                           up[1].double(), up[2].double(), bool(wb))
        s64, c64, z64 = sig.double().requires_grad_(), rgbs.double().requires_grad_(), z.double().requires_grad_()
        o = oracle.composite(s64, c64, z64, bool(wb))
        ((o[0] * up[0]).sum() + (o[1] * up[1]).sum() + (o[2] * up[2]).sum()).backward()
        assert rel_err(gs, s64.grad) < 1e-10 and rel_err(gc, c64.grad) < 1e-12 and rel_err(gz, z64.grad) < 1e-10
    rgb, dep, acc = oracle.composite(sig, rgbs, z[0], False)
    assert torch.equal(rgb, T(g["vr2_rgb"])) and torch.equal(dep, T(g["vr2_depth"])) and torch.equal(acc, T(g["vr2_acc"]))
    rgb, dep, _ = oracle.composite(torch.relu(sig), rgbs, z[0], False, use_relu=False)
    assert torch.equal(rgb, T(g["vr1_rgb"])) and torch.equal(dep, T(g["vr1_depth"]))
    rgb, dep, acc = oracle.composite(sig[:15].reshape(3, 5, 16), rgbs[:15].reshape(3, 5, 16, 3), z[:3], False)
    assert torch.equal(rgb, T(g["vrb_rgb"])) and torch.equal(dep, T(g["vrb_depth"])) and torch.equal(acc, T(g["vrb_acc"]))


def test_render_box_forward_backward():
    g = load_golden("render_box_c1")
    sd = oracle.init_codenerf_state(seed=int(g["seed"]))
    _check_weights(g, sd)
    sd = {k: v.requires_grad_() for k, v in sd.items()}
    cam = T(g["cam_pose"]).requires_grad_()
    shp, tex = T(g["shapecode"]).requires_grad_(), T(g["texturecode"]).requires_grad_()
    rgb, dep, acc, hit = oracle.render_rays_box(sd, T(g["K"]), cam, g["wlh"], g["roi"], int(g["im_sz"]), int(g["n_samples"]),
                                                shp, tex, T(g["jitter"]))
    assert np.array_equal(hit.numpy(), g["hit"]) and 0 < hit.sum() < hit.numel()
    assert rel_err(rgb, g["rgb"]) < TOL and rel_err(dep, g["depth"]) < TOL and rel_err(acc, g["acc"]) < TOL
    loss = oracle.refine_losses(rgb, acc, T(g["rgb_tgt"]), T(g["occ_pixels"]))[0]
    loss.backward()
    assert rel_err(loss, g["loss"]) < TOL
    assert rel_err(cam.grad, g["g_cam_pose"]) < 2e-5  # fp32 autograd through 1/d at grazing rays
    assert rel_err(shp.grad, g["g_shapecode"]) < 1e-5 and rel_err(tex.grad, g["g_texturecode"]) < 1e-5
    for k, v in sd.items():
        assert rel_err(v.grad, g["gw_" + k]) < 1e-5, k


def test_render_shell_forward_backward():
    g = load_golden("render_shell_c3")
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    _check_weights(g, sd)
    sd = {k: v.requires_grad_() for k, v in sd.items()}
    cam = T(g["cam_pose"]).requires_grad_()
    shp, tex = T(g["shapecode"]).requires_grad_(), T(g["texturecode"]).requires_grad_()
    rgb, dep, acc = oracle.render_rays_shell(sd, T(g["K"]), cam, g["obj_diag"], g["roi"], int(g["im_sz"]), int(g["n_samples"]),
                                             shp, tex, T(g["jitter"]))
    assert rel_err(rgb, g["rgb"]) < TOL and rel_err(dep, g["depth"]) < TOL and rel_err(acc, g["acc"]) < TOL
    loss = oracle.refine_losses(rgb, acc, T(g["rgb_tgt"]), T(g["occ_pixels"]))[0]
    loss.backward()
    assert rel_err(cam.grad, g["g_cam_pose"]) < 1e-5
    assert rel_err(shp.grad, g["g_shapecode"]) < 1e-5 and rel_err(tex.grad, g["g_texturecode"]) < 1e-5
    assert rel_err(sd["encoding_xyz.0.weight"].grad, g["gw_encoding_xyz_0_weight"]) < 1e-5
    assert rel_err(sd["encoding_viewdir.0.weight"].grad, g["gw_encoding_viewdir_0_weight"]) < 1e-5
    assert rel_err(sd["shape_latent_layer_2.0.weight"].grad, g["gw_shape_latent_layer_2_0_weight"]) < 1e-5
    assert rel_err(sd["rgb.2.weight"].grad, g["gw_rgb_2_weight"]) < 1e-5


def test_decoder_batch():
    g = load_golden("decoder_batch_c5")
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    _check_weights(g, sd)
    sd = {k: v.requires_grad_() for k, v in sd.items()}
    xyz, vd = T(g["xyz"]).requires_grad_(), T(g["viewdir"]).requires_grad_()
    B, n, S, _ = xyz.shape
    shp, tex = T(g["shapecode"]).requires_grad_(), T(g["texturecode"]).requires_grad_()
    sig, rgbs = oracle.codenerf_decoder(sd, xyz.flatten(0, 1), vd.flatten(0, 1), shp, tex)
    assert rel_err(sig, g["sigmas"]) < TOL and rel_err(rgbs, g["rgbs"]) < TOL
    rgb, dep, acc = oracle.composite(sig.reshape(B, n, S), rgbs.reshape(B, n, S, 3), T(g["z_vals"]), False)
    assert rel_err(rgb, g["rgb"]) < TOL and rel_err(acc, g["acc"]) < TOL
    oracle.refine_losses(rgb, acc, T(g["rgb_tgt"]), T(g["occ_pixels"]))[0].backward()
    assert rel_err(xyz.grad, g["g_xyz"]) < 1e-5 and rel_err(vd.grad, g["g_viewdir"]) < 1e-5
    assert rel_err(shp.grad, g["g_shapecode"]) < 1e-5 and rel_err(tex.grad, g["g_texturecode"]) < 1e-5
    for k, v in sd.items():
        assert rel_err(v.grad, g["gw_" + k]) < 1e-5, k


def test_autorf_decoder():
    g = load_golden("autorf_decoder")
    sd = oracle.init_autorf_state(seed=int(g["seed"]))
    _check_weights(g, sd)
    sd = {k: v.requires_grad_() for k, v in sd.items()}
    xyz, vd = T(g["xyz"]).requires_grad_(), T(g["viewdir"]).requires_grad_()
    shp, tex = T(g["shapecode"]).requires_grad_(), T(g["texturecode"]).requires_grad_()
    sig, rgbs = oracle.autorf_decoder(sd, xyz, vd, shp, tex)
    assert rel_err(sig, g["sigmas"]) < TOL and rel_err(rgbs, g["rgbs"]) < TOL
    ((sig * T(g["up_sigma"])).sum() + (rgbs * T(g["up_rgb"])).sum()).backward()
    assert rel_err(xyz.grad, g["g_xyz"]) < 1e-5 and rel_err(shp.grad, g["g_shapecode"]) < 1e-5
    assert rel_err(tex.grad, g["g_texturecode"]) < 1e-5 and rel_err(vd.grad, g["g_viewdir"]) < 1e-5
    for k, v in sd.items():
        assert rel_err(v.grad, g["gw_" + k]) < 1e-5, k


def test_scene_merge_oracle_matches_reference_lines():
    """oracle.merge_objects + oracle.composite against the fixture produced by executing demo.py:560-569 itself."""
    g = load_golden("scene_merge")
    z_sort, s_sort, c_sort, args = oracle.merge_objects(T(g["z_vals"]), T(g["sigmas"]), T(g["rgbs"]))
    assert np.array_equal(args.numpy(), g["z_args"]) and np.array_equal(z_sort.numpy(), g["z_sort"])
    assert np.array_equal(s_sort.numpy(), g["sigmas_sort"]) and np.array_equal(c_sort.numpy(), g["rgbs_sort"])
    rgb, dep, acc = oracle.composite(s_sort, c_sort, z_sort, white_bkgd=True)
    assert rel_err(rgb, g["rgb"]) < 1e-6 and rel_err(dep, g["depth"]) < 1e-6 and rel_err(acc, g["acc"]) < 1e-6



def test_oracle_stages_against_driver_fixture():
    """The oracle's stage functions composed the way the remaining drivers compose them, against tests/golden/drivers.npz (the
    reference's own outputs): NeRFRenderer.render_rays_specified (get_rays_specified on a non-square full-resolution crop -> box
    sampler -> decoder -> compositing, gradients to pose and codes), NeRFRenderer.prepare_pixel_samples (numpy permutation),
    NeRFRenderer.render_full_img, utils.render_rays_specified / render_full_img (shell stack) and renderer.render_rays_v3."""
    g = load_golden("drivers")
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    _check_weights(g, sd)
    K, roi_s, wlh, diag = T(g["K"]), [int(v) for v in g["roi_s"]], g["wlh"], float(g["obj_diag"])
    xs, ys = g["x_vec"] + roi_s[0], g["y_vec"] + roi_s[1]
    # NeRFRenderer.render_rays_specified (renderer.py:169-201) + the refine losses, backward
    cam = T(g["cam_pose"]).requires_grad_()
    shp, tex = T(g["shapecode"]).requires_grad_(), T(g["texturecode"]).requires_grad_()
    ro, vd = oracle.get_rays_specified(K, cam, xs, ys)
    xyz, vdr, zv, _ = oracle.prepare_sampled_rays(ro, vd, wlh, 16, T(g["rs_jitter"]))
    sig, rgbs = oracle.codenerf_decoder(sd, xyz, vdr, shp, tex)
    rgb, dep, acc = oracle.composite(sig.squeeze(-1), rgbs, zv, True)
    assert rel_err(rgb, g["rs_rgb"]) < TOL and rel_err(dep, g["rs_depth"]) < TOL and rel_err(acc, g["rs_acc"]) < TOL
    oracle.refine_losses(rgb, acc, T(g["rs_tgt"]), T(g["rs_occ"]))[0].backward()
    assert rel_err(shp.grad, g["rs_g_shp"]) < 1e-5 and rel_err(tex.grad, g["rs_g_tex"]) < 1e-5 and rel_err(cam.grad, g["rs_g_cam"]) < 1e-4
    with torch.no_grad():
        cam0, shp0, tex0 = T(g["cam_pose"]), T(g["shapecode"]), T(g["texturecode"])
        # NeRFRenderer.prepare_pixel_samples (renderer.py:203-236): the same numpy permutation under the same seed
        ro, vd = oracle.get_rays(K, cam0, roi_s)
        np.random.seed(73)
        ids = np.random.permutation(ro.shape[0])[:40]
        xyz, vdr, zv, _ = oracle.prepare_sampled_rays(ro[ids], vd[ids], wlh, 16, T(g["rp_jitter"]))
        assert rel_err(xyz, g["rp_xyz"]) < TOL and rel_err(vdr, g["rp_viewdir"]) < TOL and rel_err(zv, g["rp_z_vals"]) < TOL
        assert torch.equal(T(g["img_s"]).reshape(-1, 3)[ids], T(g["rp_tgt"])) and torch.equal(T(g["mask_s"]).reshape(-1, 1)[ids], T(g["rp_occ"]))
        # NeRFRenderer.render_full_img (renderer.py:238-294): every pixel of the crop, row-major
        xyz, vdr, zv, _ = oracle.prepare_sampled_rays(ro, vd, wlh, 16, T(g["rf_jitter"]))
        sig, rgbs = oracle.codenerf_decoder(sd, xyz, vdr, shp0, tex0)
        rgb, dep, _ = oracle.composite(sig.squeeze(-1), rgbs, zv, True)
        assert rel_err(rgb.reshape(10, 12, 3), g["rf_img"]) < TOL and rel_err(dep.reshape(10, 12), g["rf_depth"]) < TOL
        # utils.render_rays_specified (utils.py:504-551) and utils.render_full_img (:554-616): the shell stack, torch.rand(S) per call
        near, far = oracle.shell_bounds(cam0, diag)
        for seed, rays, key, shape in ((76, oracle.get_rays_specified(K, cam0, xs, ys), "us", None), (78, (ro, vd), "uf", (10, 12))):
            torch.manual_seed(seed)
            jit = torch.rand(16)
            x, v, z = oracle.sample_from_rays_shell(rays[0], rays[1], near, far, 16, jit)
            sig, rgbs = oracle.codenerf_decoder(sd, oracle.shapenet_swap(x / diag), oracle.shapenet_swap(v), shp0, tex0)
            rgb, dep, acc = oracle.composite(sig.squeeze(-1), rgbs, z.unsqueeze(0).expand(x.shape[0], -1), False)
            if shape is None:
                assert rel_err(rgb, g["us_rgb"]) < TOL and rel_err(dep, g["us_depth"]) < TOL and rel_err(acc, g["us_acc"]) < TOL
            else:
                assert rel_err(rgb.reshape(*shape, 3), g["uf_img"]) < TOL and rel_err(dep.reshape(shape), g["uf_depth"]) < TOL
        # renderer.render_rays_v3 (renderer.py:382-473): slab test on detached rays, 64 strata, adjust_scale, shapenet frame, black background
        ro, vd = oracle.get_rays(K, cam0, g["roi"], uv_steps=[8, 8])
        xyz, vdr, zv, _ = oracle.prepare_sampled_rays(ro, vd, wlh, 64, T(g["v3_jitter"]))
        sig, rgbs = oracle.codenerf_decoder(sd, oracle.shapenet_swap(xyz * 1.1), oracle.shapenet_swap(vdr), shp0, tex0)
        rgb, dep, acc = oracle.composite(sig.squeeze(-1), rgbs, zv, False)
        assert rel_err(rgb, g["v3_rgb"]) < TOL and rel_err(dep, g["v3_depth"]) < TOL and rel_err(acc, g["v3_acc"]) < TOL
