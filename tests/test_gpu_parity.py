"""GPU parity tests: every kernel, called through the reference-shaped Python API (=> ctypes => C ABI), against
the CPU oracle on identical seeded inputs and against the reference-generated golden fixtures.

Tolerances (SURVEY §8(d)): integers/bools bit-exact; floats per-tensor max|a-b|/max|b| <= 1e-5 in fp32 mode.
The weight gradients of the render_box_c1 and decoder_batch_c5 fixtures are stored as a strided sample of 1/2 .. 1/9 of their
elements (conftest.Sampled): they are judged on those elements, against max|.| of the whole array."""
import contextlib
import math

import numpy as np
import pytest
import torch

from conftest import ADAM_OUTLIERS, T, close_vs_truth, load_golden, parity_ok, rel_err
from oracle import oracle

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = "cuda"


def snb():
    import supnerf_b200
    return supnerf_b200


@contextlib.contextmanager
def forced_rand_like(value):
    """Make the next torch.rand_like return `value` (the golden/CPU jitter), so CPU oracle and GPU kernels sample
    the same strata (parity mode of SURVEY §7.3 #6)."""
    orig = torch.rand_like

    def fake(t, *a, **k):
        assert tuple(t.shape) == tuple(value.shape), (t.shape, value.shape)
        return value.to(t.device, t.dtype)
    torch.rand_like = fake
    try:
        yield
    finally:
        torch.rand_like = orig


def model_from_state(cls, sd, *args, **kw):
    m = cls(*args, **kw)
    m.load_state_dict({k: v.detach().clone() for k, v in sd.items()})
    return m.to(DEV)


# ------------------------------------------------------------------------------------------- compositing
@pytest.mark.parametrize("N,S", [(1, 2), (5, 7), (1000, 37), (4096, 64), (3000, 128), (257, 200),
                                 # the fast path with lanes left empty (8 / 16 / 32 lanes per ray) and a last warp the rays do not fill
                                 (37, 4), (77, 12), (5, 20), (1001, 36), (133, 100), (45, 124)])
@pytest.mark.parametrize("white", [False, True])
def test_composite_vs_oracle(N, S, white):
    g = torch.Generator().manual_seed(N * 131 + S)
    sig = torch.randn(N, S, generator=g) * 3
    rgbs = torch.rand(N, S, 3, generator=g) * 1.5 - 0.25
    z = torch.sort(torch.rand(N, S, generator=g) * 4 + 2, -1)[0]
    if N > 4:
        sig[1] = 1e4      # opaque everywhere: t == 1e-10 exactly
        sig[2] = -1.0     # empty
        z[3] = 2.5        # miss-ray layout: all samples at one point
    up = torch.randn(N, 3, generator=g), torch.randn(N, generator=g), torch.randn(N, generator=g)
    s_, c_, z_ = sig.clone().requires_grad_(), rgbs.clone().requires_grad_(), z.clone().requires_grad_()
    o = oracle.composite(s_, c_, z_, white)
    ((o[0] * up[0]).sum() + (o[1] * up[1]).sum() + (o[2] * up[2]).sum()).backward()
    sd, cd, zd = sig.to(DEV).requires_grad_(), rgbs.to(DEV).requires_grad_(), z.to(DEV).requires_grad_()
    r = snb().renderer.NeRFRenderer(n_samples=S, white_bkgd=white).volume_render(sd, cd, zd)
    ((r[0] * up[0].to(DEV)).sum() + (r[1] * up[1].to(DEV)).sum() + (r[2] * up[2].to(DEV)).sum()).backward()
    for a, b in zip(r, o):
        assert parity_ok("a", a, b, TOL)
    assert parity_ok("sd_grad", sd.grad, s_.grad, TOL) and parity_ok("cd_grad", cd.grad, c_.grad, TOL) and parity_ok("zd_grad", zd.grad, z_.grad, TOL)


def test_composite_golden_all_variants():
    g = load_golden("stages")
    S = snb()
    sig, rgbs, z = T(g["vr_sig"], device=DEV), T(g["vr_rgbs"], device=DEV), T(g["vr_z"], device=DEV)
    for wb in (0, 1):
        s_, c_, z_ = sig.clone().requires_grad_(), rgbs.clone().requires_grad_(), z.clone().requires_grad_()
        rgb, dep, acc = S.renderer.volume_rendering3(s_.unsqueeze(-1), c_, z_, white_bkgd=bool(wb))
        assert parity_ok("rgb", rgb, g[f"vr_rgb_wb{wb}"], TOL) and parity_ok("dep", dep, g[f"vr_depth_wb{wb}"], TOL)
        assert parity_ok("acc", acc, g[f"vr_acc_wb{wb}"], TOL)
        up = [T(g[k], device=DEV) for k in ("vr_up_rgb", "vr_up_depth", "vr_up_acc")]
        ((rgb * up[0]).sum() + (dep * up[1]).sum() + (acc * up[2]).sum()).backward()
        assert parity_ok("s__grad", s_.grad, g[f"vr_gsig_wb{wb}"], TOL) and parity_ok("c__grad", c_.grad, g[f"vr_grgb_wb{wb}"], TOL)
        assert parity_ok("z__grad", z_.grad, g[f"vr_gz_wb{wb}"], TOL)
    rgb, dep, acc = S.utils.volume_rendering2(sig.unsqueeze(-1), rgbs, z[0])
    assert parity_ok("rgb", rgb, g["vr2_rgb"], TOL) and parity_ok("dep", dep, g["vr2_depth"], TOL) and parity_ok("acc", acc, g["vr2_acc"], TOL)
    rgb, dep = S.utils.volume_rendering(torch.relu(sig).unsqueeze(-1), rgbs, z[0])
    assert parity_ok("rgb", rgb, g["vr1_rgb"], TOL) and parity_ok("dep", dep, g["vr1_depth"], TOL)
    rgb, dep, acc = S.utils.volume_rendering_batch(sig[:15].reshape(3, 5, 16, 1), rgbs[:15].reshape(3, 5, 16, 3), z[:3])
    assert parity_ok("rgb", rgb, g["vrb_rgb"], TOL) and parity_ok("dep", dep, g["vrb_depth"], TOL) and parity_ok("acc", acc, g["vrb_acc"], TOL)
    assert rgb.shape == (3, 5, 3) and acc.shape == (3, 5)


def test_composite_shared_z_gradient():
    g = torch.Generator().manual_seed(3)
    N, S = 50, 16
    sig, rgbs = torch.randn(N, S, generator=g), torch.rand(N, S, 3, generator=g)
    z = torch.sort(torch.rand(S, generator=g) * 3 + 1)[0]
    z_ = z.clone().requires_grad_()
    o = oracle.composite(sig, rgbs, z_, False)
    (o[0].sum() + 2 * o[1].sum() + o[2].sum()).backward()
    zd = z.to(DEV).requires_grad_()
    r = snb().utils.volume_rendering2(sig.to(DEV).unsqueeze(-1), rgbs.to(DEV), zd)
    (r[0].sum() + 2 * r[1].sum() + r[2].sum()).backward()
    assert parity_ok("zd_grad", zd.grad, z_.grad, TOL)


# ------------------------------------------------------------------------------------------- rays / slab / samplers
def test_get_rays_golden_and_pose_gradient():
    g = load_golden("stages")
    S = snb()
    K, c2w = T(g["K"], device=DEV), T(g["c2w"], device=DEV).requires_grad_()
    ro, vd = S.utils.get_rays(K, c2w, T(g["roi"]), uv_steps=[12, 12])
    assert torch.equal(ro.cpu(), T(g["rays_o"])) and parity_ok("vd", vd, g["viewdir"], 1e-6)
    ro2, vd2 = S.utils.get_rays(K, c2w, torch.tensor([100, 50, 109, 57], dtype=torch.int32))
    assert parity_ok("vd2", vd2, g["viewdir_full"], 1e-6) and ro2.shape == (63, 3)
    ro3, vd3 = S.utils.get_rays_specified(K, c2w, g["x_vec"] + g["roi"][0], g["y_vec"] + g["roi"][1])
    assert parity_ok("vd3", vd3, g["viewdir_spec"], 1e-6)
    w1, w2 = torch.randn(144, 3, generator=torch.Generator().manual_seed(1)), torch.randn(144, 3, generator=torch.Generator().manual_seed(2))
    ((ro * w1.to(DEV)).sum() + (vd * w2.to(DEV)).sum()).backward()
    c = T(g["c2w"]).requires_grad_()
    o = oracle.get_rays(T(g["K"]), c, g["roi"], uv_steps=[12, 12])
    ((o[0] * w1).sum() + (o[1] * w2).sum()).backward()
    assert parity_ok("c2w_grad", c2w.grad, c.grad, TOL)


def test_slab_hit_mask_bit_exact_golden():
    g = load_golden("stages")
    S = snb()
    o, d, half = g["box_o"], g["box_d"], g["box_half"]
    n = o.shape[0]
    amin, amax = np.repeat(-half[None], n, 0), np.repeat(half[None], n, 0)
    zi, zo, hit = S.utils.ray_box_intersection_tensor(T(o, device=DEV), T(d, device=DEV), T(amin, device=DEV), T(amax, device=DEV))
    assert np.array_equal(hit.cpu().numpy(), g["box_hit_t"])
    assert np.array_equal(zi.cpu().numpy(), g["box_zin_t"]) and np.array_equal(zo.cpu().numpy(), g["box_zout_t"])
    zi, zo, hit = S.utils.ray_box_intersection(o, d, amin, amax)  # numpy twin
    assert np.array_equal(hit, g["box_hit_np"]) and np.array_equal(zi, g["box_zin_np"]) and np.array_equal(zo, g["box_zout_np"])
    zi, zo, hit = S.utils.ray_box_intersection_tensor(T(o, device=DEV), T(d, device=DEV))
    assert np.array_equal(hit.cpu().numpy(), g["box_hit_unit"]) and np.array_equal(zi.cpu().numpy(), g["box_zin_unit"])


def test_slab_bit_exact_large_random_and_gradient():
    rng = np.random.RandomState(0)
    n = 200000
    o = (rng.randn(n, 3) * 2).astype(np.float32)
    d = rng.randn(n, 3).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    d[:100, 0] = 0.0  # zero direction components: inf / nan paths
    o[:50, 0] = 0.5
    half = np.asarray([0.5, 0.9, 0.3], np.float32)
    amin, amax = np.repeat(-half[None], n, 0), np.repeat(half[None], n, 0)
    tn, tf, hit = oracle.ray_box_intersection_np(o, d, amin, amax)
    S = snb()
    zi, zo, h = S.utils.ray_box_intersection_tensor(T(o, device=DEV), T(d, device=DEV), T(amin, device=DEV), T(amax, device=DEV))
    assert np.array_equal(h.cpu().numpy(), hit) and 0.02 < hit.mean() < 0.9
    assert np.array_equal(zi.cpu().numpy(), tn[hit]) and np.array_equal(zo.cpu().numpy(), tf[hit])
    # gradient of the compacted outputs
    m = 4000
    oc, dc = T(o[100:100 + m]).requires_grad_(), T(d[100:100 + m]).requires_grad_()
    a, b, hh = oracle.ray_box_intersection(oc, dc, T(amin[:m]), T(amax[:m]))
    (a[hh].sum() + 2 * b[hh].sum()).backward()
    og, dg = T(o[100:100 + m], device=DEV).requires_grad_(), T(d[100:100 + m], device=DEV).requires_grad_()
    zi, zo, _ = S.utils.ray_box_intersection_tensor(og, dg, T(amin[:m], device=DEV), T(amax[:m], device=DEV))
    (zi.sum() + 2 * zo.sum()).backward()
    assert parity_ok("og_grad", og.grad, oc.grad, TOL) and parity_ok("dg_grad", dg.grad, dc.grad, TOL)


@pytest.mark.parametrize("S_", [1, 16, 64, 100])
def test_box_sampler_vs_oracle(S_):
    obj = oracle.synthetic_object(11, im_sz=24)
    ro, vd = oracle.get_rays(obj["K"], obj["cam_pose"], obj["roi"], uv_steps=[24, 24])
    jit = torch.rand(ro.shape[0], S_, generator=torch.Generator().manual_seed(S_))
    ro_c, vd_c = ro.clone().requires_grad_(), vd.clone().requires_grad_()
    xyz, vr, zv, hit = oracle.prepare_sampled_rays(ro_c, vd_c, obj["wlh"], S_, jit)
    ws = [torch.randn(x.shape, generator=torch.Generator().manual_seed(i)) for i, x in enumerate((xyz, vr, zv))]
    ((xyz * ws[0]).sum() + (vr * ws[1]).sum() + (zv * ws[2]).sum()).backward()
    R = snb().renderer.NeRFRenderer(n_samples=S_)
    ro_g, vd_g = ro.to(DEV).requires_grad_(), vd.to(DEV).requires_grad_()
    with forced_rand_like(jit):
        xyz2, vr2, zv2, hit2 = R.prepare_sampled_rays(ro_g, vd_g, obj["wlh"])
    assert torch.equal(hit2.cpu(), hit) and 0 < hit.sum() < hit.numel()
    assert torch.equal(xyz2.cpu(), xyz.detach()), "xyz must be bit-exact (same fp32 op order)"
    assert torch.equal(vr2.cpu(), vr.detach()) and parity_ok("zv2", zv2, zv, 1e-6)
    # integer parity: the stratum index of every sample on hit rays, floor((z - near)/(far - near) * S) == k
    diag, half = oracle.box_constants(obj["wlh"])
    o_n = ro / (diag / 2)
    tn, tf, _ = oracle.ray_box_intersection(o_n, vd, -T(half).expand_as(o_n), T(half).expand_as(o_n))
    zg = ((xyz2.cpu().double() - o_n[:, None].double()) * vd[:, None].double()).sum(-1) / (vd.double() ** 2).sum(-1, keepdim=True)
    wide = hit & ((tf - tn) > 1e-3)
    kk = torch.floor((zg - tn[:, None].double()) / (tf - tn)[:, None].double() * S_ + 1e-6).long()[wide]
    assert (kk == torch.arange(S_)[None]).float().mean() > 0.999
    ((xyz2 * ws[0].to(DEV)).sum() + (vr2 * ws[1].to(DEV)).sum() + (zv2 * ws[2].to(DEV)).sum()).backward()
    assert parity_ok("ro_g_grad", ro_g.grad, ro_c.grad, 2e-5) and parity_ok("vd_g_grad", vd_g.grad, vd_c.grad, 2e-5)


def test_box_sampler_golden_c1():
    g = load_golden("render_box_c1")
    S = snb()
    ro, vd = S.utils.get_rays(T(g["K"], device=DEV), T(g["cam_pose"], device=DEV), T(g["roi"]), uv_steps=[int(g["im_sz"])] * 2)
    ro_c, vd_c = oracle.get_rays(T(g["K"]), T(g["cam_pose"]), g["roi"], uv_steps=[int(g["im_sz"])] * 2)
    R = S.renderer.NeRFRenderer(n_samples=int(g["n_samples"]))
    with forced_rand_like(T(g["jitter"])):
        xyz, vr, zv, hit = R.prepare_sampled_rays(ro_c.to(DEV), vd_c.to(DEV), g["wlh"])  # identical rays => integer parity
    assert np.array_equal(hit.cpu().numpy(), g["hit"])
    assert torch.equal(xyz.cpu(), T(g["xyz"])) and parity_ok("zv", zv, g["z_vals"], 1e-6)
    # stratum index of every sample on hit rays is bit-exact by construction of xyz; check it explicitly
    assert parity_ok("vd", vd, vd_c, 1e-6) and torch.equal(ro.cpu(), ro_c)


def test_shell_sampler_golden():
    g = load_golden("stages")
    S = snb()
    torch.manual_seed(12)
    xyz, vd, z = S.utils.sample_from_rays(T(g["rays_o"], device=DEV), T(g["viewdir"], device=DEV), 5.25, 9.75, 16)
    assert torch.equal(z.cpu(), T(g["shell_z"])) and torch.equal(xyz.cpu(), T(g["shell_xyz"]))
    _, _, zf = S.utils.sample_from_rays(T(g["rays_o"], device=DEV), T(g["viewdir"], device=DEV), 5.25, 9.75, 16, z_fixed=True)
    assert torch.equal(zf.cpu(), T(g["shell_z_fixed"]))
    rays = T(g["strat_rays"], device=DEV)
    with forced_rand_like(T(g["strat_jitter"])):
        zz = S.renderer.NeRFRenderer(n_samples=16).sample_from_ray(rays)
    assert parity_ok("zz", zz, g["strat_z"], 1e-6)


# ------------------------------------------------------------------------------------------- decoder (fp32 mode)
def _decoder_case(cls, sd, args, B, n, S_, seed, latent_dim=256):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(B * n, S_, 3, generator=g) - 0.5) * 2
    vd = torch.nn.functional.normalize(torch.randn(B * n, 1, 3, generator=g), dim=-1).repeat(1, S_, 1)
    shp, tex = oracle.synthetic_latents(seed, B, latent_dim)
    up_s, up_c = torch.randn(B * n, S_, 1, generator=g), torch.randn(B * n, S_, 3, generator=g)
    return xyz, vd, shp, tex, up_s, up_c


@pytest.mark.parametrize("blocks,B,n,S_", [((2, 1), 1, 64, 16), ((3, 1), 4, 33, 8), ((5, 5), 2, 10, 4), ((3, 1), 1, 1, 2)])
def test_decoder_fp32_vs_oracle_all_grads(blocks, B, n, S_):
    sd = oracle.init_codenerf_state(shape_blocks=blocks[0], texture_blocks=blocks[1], seed=blocks[0])
    xyz, vd, shp, tex, up_s, up_c = _decoder_case(None, sd, None, B, n, S_, seed=blocks[0] * 10 + B)
    sdg = {k: v.clone().requires_grad_() for k, v in sd.items()}
    ins = [t.clone().requires_grad_() for t in (xyz, vd, shp, tex)]
    sig, rgbs = oracle.codenerf_decoder(sdg, *ins)
    ((sig * up_s).sum() + (rgbs * up_c).sum()).backward()
    sd64 = {k: v.double().requires_grad_() for k, v in sd.items()}
    ins64 = [t.double().requires_grad_() for t in (xyz, vd, shp, tex)]
    sig64, rgbs64 = oracle.codenerf_decoder(sd64, *ins64)
    ((sig64 * up_s.double()).sum() + (rgbs64 * up_c.double()).sum()).backward()
    S = snb()
    m = model_from_state(S.CodeNeRF, sd, shape_blocks=blocks[0], texture_blocks=blocks[1])
    m.precision = "fp32"
    gin = [t.to(DEV).requires_grad_() for t in (xyz, vd, shp, tex)]
    sig2, rgbs2 = m(*gin)
    assert sig2.shape == sig.shape and rgbs2.shape == rgbs.shape
    assert parity_ok("sig2", sig2, sig, TOL) and parity_ok("rgbs2", rgbs2, rgbs, TOL)
    ((sig2 * up_s.to(DEV)).sum() + (rgbs2 * up_c.to(DEV)).sum()).backward()
    for a, b, c, name in zip(gin, ins, ins64, ("xyz", "viewdir", "shape", "texture")):
        assert close_vs_truth(a.grad, b.grad, c.grad)[0], (name, close_vs_truth(a.grad, b.grad, c.grad))
    for k, p in m.named_parameters():
        ok = close_vs_truth(p.grad, sdg[k].grad, sd64[k].grad)
        assert ok[0], (k, ok)


def test_decoder_golden_batch_c5_with_losses():
    g = load_golden("decoder_batch_c5")
    S = snb()
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    m = model_from_state(S.AutoRFMix, sd, 3, 1, 256)
    xyz, vd = T(g["xyz"], device=DEV).requires_grad_(), T(g["viewdir"], device=DEV).requires_grad_()
    B, n, S_, _ = xyz.shape
    shp, tex = T(g["shapecode"], device=DEV).requires_grad_(), T(g["texturecode"], device=DEV).requires_grad_()
    sig, rgbs = m(xyz.flatten(0, 1), vd.flatten(0, 1), shp, tex)
    assert parity_ok("sig", sig, g["sigmas"], TOL) and parity_ok("rgbs", rgbs, g["rgbs"], TOL)
    rgb, dep, acc = S.utils.volume_rendering_batch(sig.reshape(B, n, S_, 1), rgbs.reshape(B, n, S_, 3), T(g["z_vals"], device=DEV))
    assert parity_ok("rgb", rgb, g["rgb"], TOL) and parity_ok("dep", dep, g["depth"], TOL) and parity_ok("acc", acc, g["acc"], TOL)
    loss = oracle.refine_losses(rgb, acc, T(g["rgb_tgt"], device=DEV), T(g["occ_pixels"], device=DEV))[0]
    loss.backward()
    assert parity_ok("loss", loss, g["loss"], TOL)
    assert parity_ok("xyz_grad", xyz.grad, g["g_xyz"], TOL) and parity_ok("vd_grad", vd.grad, g["g_viewdir"], TOL)
    assert parity_ok("shp_grad", shp.grad, g["g_shapecode"], TOL) and parity_ok("tex_grad", tex.grad, g["g_texturecode"], TOL)
    for k, p in m.named_parameters():
        assert parity_ok("p_grad", p.grad, g["gw_" + k], TOL), k


# ------------------------------------------------------------------------------------------- end to end
def test_render_rays_box_golden_c1_end_to_end():
    """NeRFRenderer.render_rays (renderer.py:117) through the drop-in, CodeNeRF() defaults, fwd + bwd to the pose,
    the latents and every weight — against the reference's own outputs."""
    g = load_golden("render_box_c1")
    S = snb()
    sd = oracle.init_codenerf_state(seed=int(g["seed"]))
    m = model_from_state(S.CodeNeRF, sd)
    cam = T(g["cam_pose"], device=DEV).requires_grad_()
    shp, tex = T(g["shapecode"], device=DEV).requires_grad_(), T(g["texturecode"], device=DEV).requires_grad_()
    R = S.renderer.NeRFRenderer(n_samples=int(g["n_samples"]))
    with forced_rand_like(T(g["jitter"])):
        rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, T(g["img"]), T(g["mask_occ"]), cam, g["wlh"], T(g["K"], device=DEV),
                                                T(g["roi"]), shp, tex, im_sz=int(g["im_sz"]))
    assert parity_ok("tgt", tgt, g["rgb_tgt"], 1e-6) and torch.equal(occ.cpu(), T(g["occ_pixels"]))
    assert parity_ok("rgb", rgb, g["rgb"], TOL) and parity_ok("dep", dep, g["depth"], TOL) and parity_ok("acc", acc, g["acc"], TOL)
    loss = oracle.refine_losses(rgb, acc, tgt, occ)[0]
    loss.backward()
    assert parity_ok("loss", loss, g["loss"], TOL)
    # fp64 oracle = truth for the ill-conditioned reductions (pose gradient: per-ray terms 1e2-1e3x the sum)
    sd64 = {k: v.double().requires_grad_() for k, v in sd.items()}
    cam64 = T(g["cam_pose"]).double().requires_grad_()
    s64, t64 = T(g["shapecode"]).double().requires_grad_(), T(g["texturecode"]).double().requires_grad_()
    o = oracle.render_rays_box(sd64, T(g["K"]).double(), cam64, g["wlh"], g["roi"], int(g["im_sz"]), int(g["n_samples"]), s64, t64,
                               T(g["jitter"]).double())
    oracle.refine_losses(o[0], o[2], T(g["rgb_tgt"]).double(), T(g["occ_pixels"]).double())[0].backward()
    ok = close_vs_truth(cam.grad, g["g_cam_pose"], cam64.grad)
    assert ok[0], ("g_cam_pose", ok)
    for a, b, c, name in ((shp.grad, g["g_shapecode"], s64.grad, "shape"), (tex.grad, g["g_texturecode"], t64.grad, "texture")):
        ok = close_vs_truth(a, b, c)
        assert ok[0], (name, ok)
    for k, p in m.named_parameters():
        ok = close_vs_truth(p.grad, g["gw_" + k], sd64[k].grad)
        assert ok[0], (k, ok)


def test_render_rays_v2_shell_golden_c3_end_to_end():
    """utils.render_rays_v2 (utils.py:435), SUPNeRF 3/1/256 decoder, the refine-iteration render."""
    g = load_golden("render_shell_c3")
    S = snb()
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    cam = T(g["cam_pose"], device=DEV).requires_grad_()
    shp, tex = T(g["shapecode"], device=DEV).requires_grad_(), T(g["texturecode"], device=DEV).requires_grad_()
    torch.manual_seed(200)  # the CPU generator draws the shared jitter vector, as in the reference
    rgb, dep, acc, tgt, occ = S.utils.render_rays_v2(m, DEV, T(g["img"]), T(g["mask_occ"]), cam, g["obj_diag"][()], T(g["K"], device=DEV),
                                                     T(g["roi"]), int(g["n_samples"]), shp, tex, 1, 0, im_sz=int(g["im_sz"]), n_rays=None)
    assert parity_ok("rgb", rgb, g["rgb"], TOL) and parity_ok("dep", dep, g["depth"], TOL) and parity_ok("acc", acc, g["acc"], TOL)
    loss = oracle.refine_losses(rgb, acc, tgt, occ)[0]
    loss.backward()
    sd64 = {k: v.double().requires_grad_() for k, v in sd.items()}
    cam64 = T(g["cam_pose"]).double().requires_grad_()
    s64, t64 = T(g["shapecode"]).double().requires_grad_(), T(g["texturecode"]).double().requires_grad_()
    o = oracle.render_rays_shell(sd64, T(g["K"]).double(), cam64, g["obj_diag"], g["roi"], int(g["im_sz"]), int(g["n_samples"]),
                                 s64, t64, T(g["jitter"]).double())
    oracle.refine_losses(o[0], o[2], T(g["rgb_tgt"]).double(), T(g["occ_pixels"]).double())[0].backward()
    checks = [(cam.grad, g["g_cam_pose"], cam64.grad, "g_cam_pose"), (shp.grad, g["g_shapecode"], s64.grad, "shape"),
              (tex.grad, g["g_texturecode"], t64.grad, "texture"),
              (m.encoding_xyz[0].weight.grad, g["gw_encoding_xyz_0_weight"], sd64["encoding_xyz.0.weight"].grad, "enc_xyz.w"),
              (m.encoding_viewdir[0].weight.grad, g["gw_encoding_viewdir_0_weight"], sd64["encoding_viewdir.0.weight"].grad, "enc_vd.w"),
              (m.shape_latent_layer_2[0].weight.grad, g["gw_shape_latent_layer_2_0_weight"], sd64["shape_latent_layer_2.0.weight"].grad, "sl2.w"),
              (m.rgb[2].weight.grad, g["gw_rgb_2_weight"], sd64["rgb.2.weight"].grad, "rgb2.w"),
              (m.sigma[0].bias.grad, g["gw_sigma_0_bias"], sd64["sigma.0.bias"].grad, "sigma.b")]
    for a, b, c, name in checks:
        ok = close_vs_truth(a, b, c)
        assert ok[0], (name, ok)


def test_render_full_size_c1_properties():
    """Config-1 full size (64x64 rays x 64 samples): size-independent properties — miss rays render exactly the
    reference's closed form (rgb = last sample colour with white bkgd, depth = diag/2, acc = 1), the hit mask equals the
    oracle's bit for bit, weights sum <= 1, and the result equals the oracle on a 1/16 ray subsample."""
    S = snb()
    obj = oracle.synthetic_object(21, im_sz=64)
    sd = oracle.init_codenerf_state(seed=21)
    m = model_from_state(S.CodeNeRF, sd)
    shp, tex = oracle.synthetic_latents(21, 1)
    jit = torch.rand(4096, 64, generator=torch.Generator().manual_seed(21))
    R = S.renderer.NeRFRenderer(n_samples=64)
    with forced_rand_like(jit), torch.no_grad():
        rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, obj["img"], obj["mask_occ"], obj["cam_pose"].to(DEV), obj["wlh"],
                                                obj["K"].to(DEV), obj["roi"], shp.to(DEV), tex.to(DEV), im_sz=64)
    ids = torch.arange(0, 4096, 16)
    with torch.no_grad():
        o_rgb, o_dep, o_acc, o_hit = oracle.render_rays_box(sd, obj["K"], obj["cam_pose"], obj["wlh"], obj["roi"], 64, 64, shp, tex,
                                                            jit[ids], ray_ids=ids)
    assert parity_ok("rgb_ids", rgb[ids], o_rgb, TOL) and parity_ok("dep_ids", dep[ids], o_dep, TOL) and parity_ok("acc_ids", acc[ids], o_acc, TOL)
    ro, vd = oracle.get_rays(obj["K"], obj["cam_pose"], obj["roi"], uv_steps=[64, 64])
    _, _, _, hit = oracle.prepare_sampled_rays(ro, vd, obj["wlh"], 64, jit)
    miss = ~hit
    assert 0 < miss.sum() < 4096
    diag = float(np.linalg.norm(obj["wlh"]).astype(np.float32))
    assert torch.allclose(dep.cpu()[miss], torch.full((int(miss.sum()),), diag / 2), rtol=1e-6)
    assert torch.all(acc.cpu()[miss] == 1.0)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("n_rays", [None, 512])
def test_fused_render_equals_staged_ops(prec, n_rays):
    """renderer.render_rays through the fused C-ABI entry points (snb_render_fwd/bwd: one autograd node) must give the
    same bits as the staged path (one autograd node per stage): same kernels, same order."""
    S = snb()
    obj = oracle.synthetic_object(31, im_sz=32)
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=31)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    if prec == "bf16":
        m.requires_grad_(False)
    shp0, tex0 = oracle.synthetic_latents(31, 1)
    n = n_rays or 1024
    jit = torch.rand(n, 64, generator=torch.Generator().manual_seed(31))
    R = S.renderer.NeRFRenderer(n_samples=64)
    out = {}
    for fused in (True, False):
        S.renderer.FUSED_RENDER = fused
        try:
            cam = obj["cam_pose"].to(DEV).requires_grad_()
            shp, tex = shp0.to(DEV).requires_grad_(), tex0.to(DEV).requires_grad_()
            m.zero_grad()
            np.random.seed(5)
            with forced_rand_like(jit):
                rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"].to(DEV),
                                                        obj["roi"], shp, tex, im_sz=32, n_rays=n_rays)
            oracle.refine_losses(rgb, acc, tgt, occ)[0].backward()
            out[fused] = [rgb, dep, acc, tgt, occ, cam.grad, shp.grad, tex.grad]
            if prec == "fp32":
                out[fused] += [p.grad.clone() for p in m.parameters()]
        finally:
            S.renderer.FUSED_RENDER = True
    for a, b in zip(out[True][:5], out[False][:5]):
        if prec == "fp32":
            assert torch.equal(a, b)
        else:   # bf16: the fused path runs ONE decoder row per miss ray (compact.cu); the staged path S rows that differ by an ulp of z
            assert parity_ok("a", a, b, 1e-6)
    for a, b in zip(out[True][5:], out[False][5:]):   # gradients: atomics in the pose / weight reductions reorder the sums
        assert rel_err(a, b) < (1e-5 if prec == "fp32" else 1e-4)


def test_miss_ray_compaction_counts_and_accounting():
    """compact.cu through the fused bf16 render: hit mask bit-exact with the oracle, outputs equal to the dense path
    (SNB_NO_COMPACT semantics = the staged ops) on an object where most rays miss, and on one where every ray hits."""
    S = snb()
    for seed, im in ((31, 32), (100, 16)):
        obj = oracle.synthetic_object(seed, im_sz=im)
        if seed == 100:   # shrink the roi into the box: all hit
            r = obj["roi"].clone()
            cx, cy = (r[0] + r[2]) // 2, (r[1] + r[3]) // 2
            obj["roi"] = torch.tensor([cx - 2, cy - 2, cx + 2, cy + 2], dtype=r.dtype)
        sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
        m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
        m.precision = "bf16"
        m.requires_grad_(False)
        shp0, tex0 = oracle.synthetic_latents(seed, 1)
        jit = torch.rand(im * im, 64, generator=torch.Generator().manual_seed(seed))
        R = S.renderer.NeRFRenderer(n_samples=64)
        res = {}
        for fused in (True, False):
            S.renderer.FUSED_RENDER = fused
            try:
                cam = obj["cam_pose"].to(DEV).requires_grad_()
                shp, tex = shp0.to(DEV).requires_grad_(), tex0.to(DEV).requires_grad_()
                with forced_rand_like(jit):
                    rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"].to(DEV),
                                                            obj["roi"], shp, tex, im_sz=im)
                oracle.refine_losses(rgb, acc, tgt, occ)[0].backward()
                res[fused] = [rgb, dep, acc, cam.grad, shp.grad, tex.grad]
            finally:
                S.renderer.FUSED_RENDER = True
        for a, b in zip(res[True][:3], res[False][:3]):
            assert parity_ok("a", a, b, 1e-6)
        for a, b in zip(res[True][3:], res[False][3:]):
            assert parity_ok("a", a, b, 1e-4)
        ro, vd = oracle.get_rays(obj["K"], obj["cam_pose"], obj["roi"], uv_steps=[im, im])
        _, _, _, hit = oracle.prepare_sampled_rays(ro, vd, obj["wlh"], 64, jit)
        if seed == 100:
            assert bool(hit.all())


def test_fused_render_specified_equals_staged():
    S = snb()
    obj = oracle.synthetic_object(33, im_sz=48)
    sd = oracle.init_codenerf_state(seed=33)
    m = model_from_state(S.CodeNeRF, sd)
    shp0, tex0 = oracle.synthetic_latents(33, 1)
    rng = np.random.RandomState(3)
    x_vec, y_vec = rng.randint(0, 48, size=100), rng.randint(0, 48, size=100)
    jit = torch.rand(100, 64, generator=torch.Generator().manual_seed(33))
    R = S.renderer.NeRFRenderer(n_samples=64)
    roi = obj["roi"].clone()
    roi[2:] = roi[:2] + 48
    out = {}
    for fused in (True, False):
        S.renderer.FUSED_RENDER = fused
        try:
            cam = obj["cam_pose"].to(DEV).requires_grad_()
            with forced_rand_like(jit):
                r = R.render_rays_specified(m, DEV, obj["img"], obj["mask_occ"], cam, obj["wlh"], obj["K"].to(DEV), roi, x_vec, y_vec,
                                            shp0.to(DEV), tex0.to(DEV))
            (r[0].sum() + r[1].sum() + r[2].sum()).backward()
            out[fused] = list(r) + [cam.grad]
        finally:
            S.renderer.FUSED_RENDER = True
    for a, b in zip(out[True][:5], out[False][:5]):
        assert torch.equal(a, b)
    assert parity_ok("out_True_5", out[True][5], out[False][5], 1e-5)


@pytest.mark.parametrize("n", [1, 257, 16384])
def test_refine_loss_kernel_vs_oracle(n):
    """losses.refine_loss (csrc/loss.cu) against the reference's inline loss (optimizer_nuscenes.py:729-736, restated in
    oracle.refine_losses): values and gradients, incl. a caller-supplied denominator."""
    S = snb()
    g = torch.Generator().manual_seed(n)
    rgb, tgt = torch.rand(n, 3, generator=g), torch.rand(n, 3, generator=g)
    acc = torch.rand(n, generator=g)
    occ = torch.randint(-1, 2, (n, 1), generator=g).float()
    if n == 1:
        occ[:] = 1.0
    r64, a64 = rgb.double().requires_grad_(), acc.double().requires_grad_()
    l64 = oracle.refine_losses(r64, a64, tgt.double(), occ.double())
    l64[0].backward()
    r, a = rgb.to(DEV).requires_grad_(), acc.to(DEV).requires_grad_()
    loss, l_rgb, l_occ = S.losses.refine_loss(r, a, tgt.to(DEV), occ.to(DEV), 0.1)
    (3.0 * loss).backward()
    assert parity_ok("loss", loss, l64[0], TOL) and parity_ok("l_rgb", l_rgb, l64[1], TOL) and parity_ok("l_occ", l_occ, l64[2], TOL)
    assert parity_ok("r_grad", r.grad, 3.0 * r64.grad, TOL) and parity_ok("a_grad", a.grad, 3.0 * a64.grad, TOL)
    # caller-supplied (global) denominator: the ray-sharded partial loss
    den = torch.tensor([2.0 * occ.abs().sum().item() + 1e-9], device=DEV)
    half = S.losses.refine_loss(rgb.to(DEV), acc.to(DEV), tgt.to(DEV), occ.to(DEV), 0.1, den=den)[0]
    assert parity_ok("half", half, 0.5 * l64[0], TOL)
    # B objects in one launch per direction (refine_loss_batch) against the per-object entry point on the same rows: the fp64 sums
    # may be added in another order, the gradients are the same arithmetic bit for bit
    B = 3
    rgb_b, tgt_b, acc_b = torch.rand(B, n, 3, generator=g), torch.rand(B, n, 3, generator=g), torch.rand(B, n, generator=g)
    occ_b = torch.randint(-1, 2, (B, n, 1), generator=g).float()
    if n == 1:
        occ_b[:] = 1.0
    rb, ab = rgb_b.to(DEV).requires_grad_(), acc_b.to(DEV).requires_grad_()
    loss_b, parts_b = S.losses.refine_loss_batch(rb, ab, tgt_b.to(DEV), occ_b.to(DEV), 0.1)
    (3.0 * loss_b).sum().backward()
    for i in range(B):
        ri, ai = rgb_b[i].to(DEV).requires_grad_(), acc_b[i].to(DEV).requires_grad_()
        li, vec = S.losses.refine_loss_vec(ri, ai, tgt_b[i].to(DEV), occ_b[i].to(DEV), 0.1)
        (3.0 * li).backward()
        torch.testing.assert_close(parts_b[i], vec, rtol=1e-6, atol=0)
        assert torch.equal(rb.grad[i], ri.grad) and torch.equal(ab.grad[i], ai.grad)
    with pytest.raises(S._lib.SnbError):
        S.losses.refine_loss(rgb, acc, tgt, occ)   # CPU tensors: no fallback


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("n_rays,sym", [(None, 0), (512, 1)])
def test_fused_shell_render_equals_staged_ops(prec, n_rays, sym):
    """utils.render_rays_v2 (the refine loops' render, utils.py:435) through the fused C-ABI entry points in shell mode vs
    the staged ops: same bits forward (same kernels), gradients to 1e-5; with sym_aug the flip draw must be consumed alike."""
    import random
    S = snb()
    obj = oracle.synthetic_object(35, im_sz=32)
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=35)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    if prec == "bf16":
        m.requires_grad_(False)
    shp0, tex0 = oracle.synthetic_latents(35, 1)
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    out = {}
    for fused in (True, False):
        S.utils.FUSED_RENDER = fused
        try:
            for trial in range(3 if sym else 1):   # several draws so that both flip outcomes occur
                cam = obj["cam_pose"].to(DEV).requires_grad_()
                shp, tex = shp0.to(DEV).requires_grad_(), tex0.to(DEV).requires_grad_()
                m.zero_grad()
                np.random.seed(5 + trial); torch.manual_seed(9 + trial); random.seed(11 + trial)
                rgb, dep, acc, tgt, occ = S.utils.render_rays_v2(m, DEV, obj["img"], obj["mask_occ"], cam, diag, obj["K"].to(DEV), obj["roi"],
                                                                 64, shp, tex, 1, sym, im_sz=32, n_rays=n_rays)
                oracle.refine_losses(rgb, acc, tgt, occ)[0].backward()
                out[(fused, trial)] = [rgb, dep, acc, tgt, occ, cam.grad, shp.grad, tex.grad]
        finally:
            S.utils.FUSED_RENDER = True
    for (fused, trial), vals in out.items():
        if not fused:
            continue
        ref = out[(False, trial)]
        for a, b in zip(vals[:5], ref[:5]):
            assert torch.equal(a, b)
        for a, b in zip(vals[5:], ref[5:]):
            assert parity_ok("a", a, b, 1e-5)


def test_object_refiner_matches_reference_api_loop_and_graph_replay():
    """refine.ObjectRefiner (device-side shell bounds, capturable AdamW, optional CUDA graph) against the loop written with
    the reference-shaped API (render_rays_v2 with host-side near/far + the inline losses + torch AdamW), 6 iterations."""
    S = snb()
    import tools.refine_bench as rb
    obj = oracle.synthetic_object(51, im_sz=32)
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=51)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.requires_grad_(False)
    shp0, tex0 = oracle.synthetic_latents(51, 1)
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    c2o = obj["cam_pose"]
    R_obj = c2o[:, :3].t().contiguous()
    t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
    rv0 = rb.matrix_to_axis_angle(R_obj)
    iters = 6
    # reference-API loop
    shp, tex = shp0.to(DEV).requires_grad_(), tex0.to(DEV).requires_grad_()
    rv, tv = rv0.to(DEV).requires_grad_(), t_obj.to(DEV).requires_grad_()
    opt = torch.optim.AdamW([{"params": shp, "lr": 0.02}, {"params": tex, "lr": 0.02}, {"params": rv, "lr": 0.01}, {"params": tv, "lr": 0.01}])
    # 37 "lidar" pixels inside the crop (an odd count: the refiner pads to the decoder's tile); the crop is rendered at im_sz = 32 from a
    # roi of another size, render_rays_specified addresses full-resolution pixels of the crop
    roi_t = torch.as_tensor(np.asarray(obj["roi"]))
    gl = np.random.RandomState(5)
    h_c, w_c = obj["img"].shape[0], obj["img"].shape[1]
    ly, lx = gl.randint(0, h_c, 37), gl.randint(0, w_c, 37)
    torch.manual_seed(77)
    for _ in range(iters):
        opt.zero_grad()
        rot = S.refine.axis_angle_to_matrix(rv).t()
        cam = torch.cat((rot, -rot @ tv.unsqueeze(-1)), -1)
        rgb, dep, acc, tgt, occ = S.utils.render_rays_v2(m, DEV, obj["img"], obj["mask_occ"], cam, diag, obj["K"].to(DEV), obj["roi"], 64,
                                                         shp, tex, 1, 0, im_sz=32, n_rays=None)
        loss_ref = oracle.refine_losses(rgb, acc, tgt, occ)[0]
        loss_ref.backward()
        # the per-iteration evaluation of optimizer_nuscenes.py:740-769: PSNR loss over the object mask, lidar-pixel depth render
        mask_rgb = occ.clone()
        mask_rgb[occ < 0] = 0
        loss_rgb2_ref = torch.sum((rgb - tgt) ** 2 * mask_rgb) / (torch.sum(mask_rgb) + 1e-9)
        with torch.no_grad():
            _, depth_ref, _, _, _ = S.utils.render_rays_specified(m, DEV, obj["img"], obj["mask_occ"], cam, diag, obj["K"].to(DEV), roi_t, lx, ly,
                                                                  64, shp, tex, 1, 0)
        opt.step()
    outs = []
    for graphed, fused in ((False, False), (True, False), (False, True), (True, True)):
        torch.manual_seed(77)   # the refiner pre-draws the same torch.rand(64) sequence
        r = S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], diag, shp0, tex0, rv0, t_obj, n_samples=64,
                                   im_sz=32, max_iters=iters, fused=fused, lidar_xy=(lx, ly))
        if graphed:
            r.capture()
        last = r.run(iters)
        torch.cuda.synchronize()
        outs.append((r, last.clone()))
        assert parity_ok("last_0", last[0], loss_ref, 1e-4)
        assert parity_ok("loss_rgb2", r.loss_rgb2, loss_rgb2_ref, 1e-4)
        assert r.depth_pred.shape == depth_ref.shape and parity_ok("lidar_depth", r.depth_pred, depth_ref, 1e-4)
        # Adam's g / sqrt(v) turns last-ulp differences of near-zero gradient components into O(lr) parameter differences:
        # the codes are compared at 2e-2 of their scale, the loss trajectory and the (well-conditioned) pose tightly
        assert parity_ok("r_shapecode", r.shapecode, shp, 2e-2, outliers=ADAM_OUTLIERS) and parity_ok("r_texturecode", r.texturecode, tex, 2e-2, outliers=ADAM_OUTLIERS)
        assert parity_ok("r_rot_vec", r.rot_vec, rv, 1e-3) and parity_ok("r_trans_vec", r.trans_vec, tv, 1e-3)
    for o in outs[1:]:
        assert parity_ok("o_0_shapecode", o[0].shapecode, outs[0][0].shapecode, 2e-2, outliers=ADAM_OUTLIERS) and parity_ok("o_1", o[1], outs[0][1], 1e-4)


@pytest.mark.parametrize("prec,tol_loss", [("fp32", 1e-3), ("bf16", 5e-3)])
def test_object_refiner_50_iterations_loss_trajectory(prec, tol_loss):
    """The metric "ms per refine iteration" is quoted on 50 iterations: the graphed ObjectRefiner against the loop written with the
    reference-shaped API (utils.render_rays_v2 with its host-side near / far + the inline losses of optimizer_nuscenes.py:729-736 +
    torch.optim.AdamW), same seed, 50 iterations -- the loss of EVERY iteration within 1e-3 (relative to the loop's) in fp32 mode and
    5e-3 in bf16 mode (both loops run the same kernels; the decoder's atomically accumulated latent sums differ in the last bit from run
    to run and Adam's g / sqrt(v) amplifies that over 50 steps: 6e-5 .. 1e-3 measured; the mode's own budget is 2e-2), the final pose
    within 5e-3.  Recorded beside it (information only): the distance of the trajectory from the fp32 CPU oracle's loop."""
    from conftest import parity
    S = snb()
    import tools.refine_bench as rb
    obj = oracle.synthetic_object(53, im_sz=32)
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=53)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    m.requires_grad_(False)
    shp0, tex0 = oracle.synthetic_latents(53, 1)
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    c2o = obj["cam_pose"]
    R_obj = c2o[:, :3].t().contiguous()
    t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
    rv0 = rb.matrix_to_axis_angle(R_obj)
    iters = 50
    lrs = (0.02, 0.02, 0.01, 0.01)

    def api_loop(render, dev, model_or_sd):
        shp, tex = shp0.to(dev).requires_grad_(), tex0.to(dev).requires_grad_()
        rv, tv = rv0.to(dev).requires_grad_(), t_obj.to(dev).requires_grad_()
        opt = torch.optim.AdamW([{"params": p_, "lr": lr} for p_, lr in zip((shp, tex, rv, tv), lrs)])
        torch.manual_seed(79)
        traj = []
        for _ in range(iters):
            opt.zero_grad()
            rot = S.refine.axis_angle_to_matrix(rv).t()
            cam = torch.cat((rot, -rot @ tv.unsqueeze(-1)), -1)
            rgb, acc, tgt, occ = render(model_or_sd, cam, shp, tex)
            loss = oracle.refine_losses(rgb, acc, tgt, occ)[0]
            loss.backward()
            opt.step()
            traj.append(loss.detach().cpu())
        return torch.stack(traj), rv.detach().cpu(), tv.detach().cpu()

    def render_gpu(model, cam, shp, tex):
        rgb, dep, acc, tgt, occ = S.utils.render_rays_v2(model, DEV, obj["img"], obj["mask_occ"], cam, diag, obj["K"].to(DEV), obj["roi"], 64,
                                                         shp, tex, 1, 0, im_sz=32, n_rays=None)
        return rgb, acc, tgt, occ

    traj_api, rv_api, tv_api = api_loop(render_gpu, DEV, m)
    torch.manual_seed(79)   # the refiner pre-draws the same torch.rand(64) sequence
    r = S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], diag, shp0, tex0, rv0, t_obj, n_samples=64,
                               im_sz=32, max_iters=iters).capture()
    traj = []
    for _ in range(iters):
        traj.append(r.run(1)[0].clone())
    traj = torch.stack(traj).cpu()
    worst = float(((traj - traj_api).abs() / traj_api.abs()).max())
    parity("loss_trajectory_50_iterations_vs_reference_api_loop", traj, traj_api, tol_loss)
    assert worst <= tol_loss, worst                       # every iteration, relative to that iteration's loss
    assert float(traj[-1]) < float(traj[0])               # and it optimises
    # Adam's g / sqrt(v) turns last-ulp differences of near-zero gradient components (atomics reorder the sums) into O(lr)
    # parameter differences that accumulate over 50 steps: the pose is compared at 5e-3, the loss of every iteration at 1e-3
    parity("rot_vec_after_50", r.rot_vec, rv_api, 5e-3)
    parity("trans_vec_after_50", r.trans_vec, tv_api, 5e-3)
    if prec == "fp32":
        def render_cpu(sd_, cam, shp, tex):
            jit = torch.rand(64)
            rgb, dep, acc = oracle.render_rays_shell(sd_, obj["K"], cam, diag, obj["roi"], 32, 64, shp, tex, jit)
            return rgb, acc, obj["img"].reshape(-1, 3), obj["mask_occ"].reshape(-1, 1)
        traj_o, _, _ = api_loop(render_cpu, "cpu", sd)
        parity("loss_trajectory_50_iterations_vs_fp32_cpu_oracle_loop", traj, traj_o, tol_loss, info=True)


def test_run_objects_side_by_side_equals_one_after_the_other():
    """refine.run_objects (independent objects' graph replays issued round-robin over several CUDA streams) leaves every object
    in the state its own sequential loop would: same kernels, same order per object, no shared mutable state."""
    S = snb()
    import tools.refine_bench as rb
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=52)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.requires_grad_(False)
    iters = 5

    def make(seed):
        obj = oracle.synthetic_object(seed, im_sz=32)
        shp0, tex0 = oracle.synthetic_latents(seed, 1)
        c2o = obj["cam_pose"]
        R_obj = c2o[:, :3].t().contiguous()
        t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
        torch.manual_seed(seed)
        return S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                      shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, n_samples=64, im_sz=32, max_iters=iters).capture()

    seq = [make(60 + k) for k in range(3)]
    for r in seq:
        r.run(iters)
    par = [make(60 + k) for k in range(3)]
    S.refine.run_objects(par, iters, n_streams=3)
    torch.cuda.synchronize()
    for a, b in zip(seq, par):
        # (the decoder's latent-gradient column sums are accumulated with atomics: equal to rounding, not bit for bit)
        assert parity_ok("b_loss", b.loss, a.loss, 1e-4)
        assert parity_ok("b_shapecode", b.shapecode, a.shapecode, 2e-2, outliers=ADAM_OUTLIERS) and parity_ok("b_texturecode", b.texturecode, a.texturecode, 2e-2, outliers=ADAM_OUTLIERS)
        assert parity_ok("b_rot_vec", b.rot_vec, a.rot_vec, 1e-3) and parity_ok("b_trans_vec", b.trans_vec, a.trans_vec, 1e-3)


def test_device_side_shell_samples_match_host_built_vector():
    """refine.shell_samples_on_device vs the reference's host arithmetic (utils.py:154-167, :468-469)."""
    S = snb()
    for seed in range(5):
        obj = oracle.synthetic_object(60 + seed, im_sz=8)
        diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
        jit = torch.rand(64, generator=torch.Generator().manual_seed(seed))
        near, far = oracle.shell_bounds(obj["cam_pose"], float(diag))
        dist = (far - near) / (2 * 64)
        z_ref = torch.linspace(near + dist, far - dist, 64) + jit * (far - near) / (2 * 64)
        z = S.refine.shell_samples_on_device(obj["cam_pose"].to(DEV), diag, 64, jit.to(DEV))
        assert parity_ok("z", z, z_ref, 2e-7)


def test_scene_merge_kernel_golden_and_random():
    """scene.merge_objects / render_merged (csrc/scene.cu) against the reference's own lines (fixture) and the oracle on a
    larger random case with many ties: the searchsorted indices and the scattered values bit-exact, the render to 1e-5."""
    S = snb()
    g = load_golden("scene_merge")
    zs, ss, cs, args = S.scene.merge_objects(T(g["z_vals"], device=DEV), T(g["sigmas"], device=DEV), T(g["rgbs"], device=DEV), return_args=True)
    assert np.array_equal(args.cpu().numpy(), g["z_args"]) and np.array_equal(zs.cpu().numpy(), g["z_sort"])
    assert np.array_equal(ss.cpu().numpy(), g["sigmas_sort"]) and np.array_equal(cs.cpu().numpy(), g["rgbs_sort"])
    rgb, dep, acc = S.scene.render_merged(T(g["z_vals"], device=DEV), T(g["sigmas"], device=DEV), T(g["rgbs"], device=DEV))
    assert parity_ok("rgb", rgb, g["rgb"], TOL) and parity_ok("dep", dep, g["depth"], TOL) and parity_ok("acc", acc, g["acc"], TOL)
    gen = torch.Generator().manual_seed(3)
    R_, Nb, S_ = 3000, 8, 64                                   # K = 512 samples per ray
    z = (torch.rand(R_, Nb, S_, generator=gen) * 20).round() / 4      # quantised depths: many ties
    z[torch.rand(R_, Nb, 1, generator=gen).expand(-1, -1, S_) < 0.4] = -1.0
    z = z.reshape(R_, Nb * S_)
    sig, col = torch.rand(R_, Nb * S_, generator=gen), torch.rand(R_, Nb * S_, 3, generator=gen)
    o = oracle.merge_objects(z, sig, col)
    k = S.scene.merge_objects(z.to(DEV), sig.to(DEV), col.to(DEV), return_args=True)
    for a, b in zip(k, o):
        assert torch.equal(a.cpu(), b)
    with pytest.raises(S._lib.SnbError):
        S.scene.merge_objects(z, sig, col)     # CPU tensors: no fallback


def test_one_row_refine_pose_and_adamw_kernels_vs_torch():
    """csrc/refine.cu: the Rodrigues pose map (both conventions) + its backward against torch autograd in float64, the fused
    sample vector against refine.shell_samples_on_device, and the fused AdamW against torch.optim.AdamW over 5 steps."""
    S = snb()
    gen = torch.Generator().manual_seed(9)
    for opt_cam in (False, True):
        for scale in (1.3, 1e-5):           # generic angle and the small-angle series
            rv = (torch.randn(3, generator=gen) * scale)
            tv = torch.randn(3, generator=gen) * 5
            jit = torch.rand(64, generator=gen)
            up = torch.randn(3, 4, generator=gen)
            r64, t64 = rv.double().requires_grad_(), tv.double().requires_grad_()
            rot = S.refine.axis_angle_to_matrix(r64)
            tt = t64.unsqueeze(-1)
            if not opt_cam:
                rot = rot.transpose(-2, -1)
                tt = -rot @ tt
            cam64 = torch.cat((rot, tt), -1)
            (cam64 * up.double()).sum().backward()
            rg, tg = rv.to(DEV).requires_grad_(), tv.to(DEV).requires_grad_()
            one = torch.ones(1, device=DEV, dtype=torch.uint8)
            cam, z = S.refine._PoseAndSamplesBatch.apply(rg.view(1, 3), tg.view(1, 3), jit.to(DEV).view(1, 1, 64), None,
                                                         torch.zeros(1, device=DEV), torch.tensor([4.7], device=DEV), opt_cam, 64, one)
            cam, z = cam.view(3, 4), z.view(64)
            (cam * up.to(DEV)).sum().backward()
            assert parity_ok("cam", cam, cam64, 1e-6)
            assert parity_ok("rg_grad", rg.grad, r64.grad, 1e-5) and parity_ok("tg_grad", tg.grad, t64.grad, 1e-5)
            z_ref = S.refine.shell_samples_on_device(cam.detach(), np.float32(4.7), 64, jit.to(DEV))
            assert parity_ok("z", z, z_ref, 2e-7)
    ps = [torch.randn(n, generator=gen) for n in (256, 256, 3, 3)]
    lrs = [0.02, 0.02, 0.01, 0.01]
    ref = [p.clone().requires_grad_() for p in ps]
    opt = torch.optim.AdamW([{"params": [p], "lr": lr} for p, lr in zip(ref, lrs)])
    mine = [p.to(DEV).clone().requires_grad_() for p in ps]
    fo = S.refine.SlotAdamW([{"params": p, "lr": lr} for p, lr in zip(mine, lrs)], rows=1)
    for it in range(5):
        gs = [torch.randn(p.shape, generator=gen) for p in ps]
        for p, q, g in zip(ref, mine, gs):
            p.grad = g.clone()
            q.grad = g.to(DEV)
        opt.step()
        fo.step()
    for p, q in zip(ref, mine):
        assert parity_ok("q", q, p, 1e-6)



def test_shell_sample_vector_on_device_option():
    """utils.SHELL_Z_ON_DEVICE: the reference-shaped shell drivers without the per-call device -> host read of the pose; renders equal
    to the default (host-built vector) path to 1e-5, and no synchronisation is needed to issue the call."""
    S = snb()
    obj = oracle.synthetic_object(57, im_sz=16)
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=57)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = "fp32"
    m.requires_grad_(False)
    shp, tex = oracle.synthetic_latents(57, 1)
    diag = np.linalg.norm(obj["wlh"]).astype(np.float32)
    outs = []
    try:
        for flag in (False, True):
            S.utils.SHELL_Z_ON_DEVICE = flag
            torch.manual_seed(3)
            cam = obj["cam_pose"].to(DEV)
            outs.append(S.utils.render_rays_v2(m, DEV, obj["img"], obj["mask_occ"], cam, diag, obj["K"].to(DEV), obj["roi"], 64, shp.to(DEV),
                                               tex.to(DEV), 1, 0, im_sz=16, n_rays=None)[:3])
    finally:
        S.utils.SHELL_Z_ON_DEVICE = False
    for a, b, n_ in zip(outs[1], outs[0], ("rgb", "depth", "acc")):
        assert parity_ok(n_, a, b, 1e-5)


@pytest.mark.parametrize("sym_aug,im_sz", [(0, 24), (1, 16)])
def test_prepare_pixel_samples_batch_equals_per_object_calls(sym_aug, im_sz):
    """SURVEY 8f rank 3: utils.prepare_pixel_samples_batch (ONE kernel for the batch, on the device) against B calls of
    utils.prepare_pixel_samples (the reference's per-object DataLoader work, utils.py:330-377) under the same RNG state: bit-identical
    samples, targets and masks, including the symmetric-augmentation flip and the shapenet swap."""
    import random
    S = snb()
    B, n_rays, S_ = 4, 200, 16
    objs = [oracle.synthetic_object(400 + i, im_sz=24) for i in range(B)]
    diags = [np.linalg.norm(o["wlh"]).astype(np.float32) for o in objs]

    def seed():
        np.random.seed(13); torch.manual_seed(13); random.seed(13)
    seed()
    per = [S.utils.prepare_pixel_samples(o["img"].to(DEV), o["mask_occ"].to(DEV), o["cam_pose"].to(DEV), d, o["K"].to(DEV), o["roi"], n_rays, S_, 1,
                                         sym_aug, im_sz=im_sz) for o, d in zip(objs, diags)]
    seed()
    xyz, vd, z, tgt, occ = S.utils.prepare_pixel_samples_batch(DEV, [o["img"] for o in objs], [o["mask_occ"] for o in objs],
                                                               [o["cam_pose"] for o in objs], diags, [o["K"] for o in objs],
                                                               [o["roi"] for o in objs], n_rays, S_, 1, sym_aug, im_sz=im_sz)
    assert xyz.shape == (B, n_rays, S_, 3) and vd.shape == xyz.shape and z.shape == (B, S_) and tgt.shape == (B, n_rays, 3)
    for i in range(B):
        assert torch.equal(xyz[i], per[i][0]) and torch.equal(vd[i], per[i][1]) and torch.equal(z[i], per[i][2].to(z.device))
        assert torch.equal(tgt[i], per[i][3].to(tgt.device)) and torch.equal(occ[i], per[i][4].to(occ.device))


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_scene_compositor_against_the_reference_vis_scene(prec):
    """SURVEY 8f rank 4: scene.render_scene (ray bookkeeping around the merge, decoder over all objects' rows, merge-sort + white
    compositing kernels) against the canvas the reference's own vis_scene (scripts/demo.py:425-579, executed unmodified by
    tools/make_golden.py:golden_scene) painted for the same three objects, camera manipulation and jitter draws.  The canvas is
    uint8: the reference evaluates the slab test in float64 on the host, the kernel in fp32, so single pixels may differ by one
    grey level (fp32 mode) / a few (bf16 mode: 2e-2 x 255 = 5)."""
    S = snb()
    g = load_golden("scene")
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"]))
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    m.requires_grad_(False)
    canvas = S.scene.render_scene(m, DEV, T(g["K"]), T(g["obj_poses"]), T(g["obj_wlh"]), T(g["shapecodes"]), T(g["texturecodes"]), int(g["H"]),
                                  int(g["W"]), int(g["n_samples"]), manipulation=[float(v) for v in g["manipulation"]], rend_aabb=True,
                                  adjust_scale=float(g["adjust_scale"]), shapenet_obj_cood=True, ray_batch_size=int(g["ray_batch_size"]),
                                  jitter=T(g["jitter"]))
    ref = g["canvas"]
    assert canvas.shape == ref.shape and canvas.dtype == np.uint8
    covered_ref, covered = (ref != 255).any(-1), (canvas != 255).any(-1)
    assert np.array_equal(covered, covered_ref)                       # the same pixels are covered by an object
    diff = np.abs(canvas.astype(np.int32) - ref.astype(np.int32))
    tol = 1 if prec == "fp32" else 5
    frac = float((diff <= tol).mean())
    from conftest import parity
    parity("canvas_uint8", canvas.astype(np.float32), ref.astype(np.float32), 1e-2 if prec == "fp32" else 2e-2)
    assert frac >= 0.999, (frac, int(diff.max()))


def test_object_group_one_graph_equals_sequential_refiners():
    """refine.ObjectGroup (all objects' iterations forked / joined inside ONE captured CUDA graph) leaves every object in the state
    its own sequential loop would."""
    S = snb()
    import tools.refine_bench as rb
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=52)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.requires_grad_(False)
    iters = 5

    def make(seed):
        obj = oracle.synthetic_object(seed, im_sz=32)
        shp0, tex0 = oracle.synthetic_latents(seed, 1)
        c2o = obj["cam_pose"]
        R_obj = c2o[:, :3].t().contiguous()
        t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
        torch.manual_seed(seed)
        return S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                      shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, n_samples=64, im_sz=32, max_iters=iters)
    seq = [make(70 + k).capture() for k in range(3)]
    for r in seq:
        r.run(iters)
    grp = S.refine.ObjectGroup([make(70 + k) for k in range(3)]).capture()
    grp.run(iters)
    torch.cuda.synchronize()
    for a, b in zip(seq, grp.refiners):
        assert parity_ok("b_loss", b.loss, a.loss, 1e-4)
        assert parity_ok("b_shapecode", b.shapecode, a.shapecode, 2e-2, outliers=ADAM_OUTLIERS) and parity_ok("b_rot_vec", b.rot_vec, a.rot_vec, 1e-3)


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_batch_refiner_one_launch_set_equals_per_object_refiners(prec):
    """refine.BatchRefiner (B objects' refine iterations as ONE launch set: batched pose map, shell render, losses, AdamW; config C3's
    per-GPU share) against every object's own ObjectRefiner loop: per-iteration losses, the masked PSNR loss, lidar-pixel depths
    (ragged pixel counts, one object without any), and the optimised codes / pose parameters."""
    S = snb()
    import tools.refine_bench as rb
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=53)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    m.requires_grad_(False)
    iters = 6
    n_lidar = [37, 0, 64, 5]

    def make(k):
        seed = 80 + k
        obj = oracle.synthetic_object(seed, im_sz=32)
        shp0, tex0 = oracle.synthetic_latents(seed, 1)
        c2o = obj["cam_pose"]
        R_obj = c2o[:, :3].t().contiguous()
        t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
        rng = np.random.RandomState(seed)
        roi = [int(v) for v in obj["roi"]]
        xy = None
        if n_lidar[k]:
            xy = (rng.randint(0, roi[2] - roi[0], n_lidar[k]), rng.randint(0, roi[3] - roi[1], n_lidar[k]))
        torch.manual_seed(seed)
        return S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                      shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, n_samples=64, im_sz=32, max_iters=iters, lidar_xy=xy)
    seq = [make(k) for k in range(4)]
    bat = S.refine.BatchRefiner([make(k) for k in range(4)])
    tol1 = 1e-5 if prec == "fp32" else 1e-4       # one iteration: same kernels on the same rows; only summation orders differ
    for it in range(iters):
        for r in seq:
            r.run(1)
        bat.run(1)
        torch.cuda.synchronize()
        tol = tol1 if it == 0 else (1e-3 if prec == "fp32" else 5e-3)     # later: the trajectories' own sensitivity (see the 50-iteration test)
        for b, r in enumerate(seq):
            assert parity_ok("it%d_loss" % it, bat.loss[b], r.loss, tol)
            assert parity_ok("it%d_loss_rgb2" % it, bat.loss_rgb2[b], r.loss_rgb2, tol)
            d = bat.lidar_depths()[b]
            if n_lidar[b]:
                assert d.shape == r.depth_pred.shape and parity_ok("it%d_lidar_depth" % it, d, r.depth_pred, tol)
            else:
                assert d is None
            if it == 0:
                # the gradients themselves (AdamW's first step is ~ lr * sign(g): an element whose gradient is at rounding level may
                # legitimately land 2 lr apart in two summation orders, so the updated codes are held to the trajectory tolerance)
                assert parity_ok("it0_g_shapecode", bat.shapecode.grad[b], r.shapecode.grad.reshape(-1), tol1)
                assert parity_ok("it0_g_texturecode", bat.texturecode.grad[b], r.texturecode.grad.reshape(-1), tol1)
                assert parity_ok("it0_g_rot_vec", bat.rot_vec.grad[b], r.rot_vec.grad, 10 * tol1)
                assert parity_ok("it0_g_trans_vec", bat.trans_vec.grad[b], r.trans_vec.grad, 10 * tol1)
                assert parity_ok("it0_shapecode", bat.shapecode[b], r.shapecode.reshape(-1), 2e-2, outliers=ADAM_OUTLIERS)
                assert parity_ok("it0_rot_vec", bat.rot_vec[b], r.rot_vec, 5e-3) and parity_ok("it0_trans_vec", bat.trans_vec[b], r.trans_vec, 5e-3)
    for b, r in enumerate(bat.write_back()):
        assert parity_ok("end_shapecode", r.shapecode, seq[b].shapecode, 2e-2, outliers=ADAM_OUTLIERS) and parity_ok("end_texturecode", r.texturecode, seq[b].texturecode, 2e-2, outliers=ADAM_OUTLIERS)
        assert parity_ok("end_rot_vec", r.rot_vec, seq[b].rot_vec, 5e-3) and parity_ok("end_trans_vec", r.trans_vec, seq[b].trans_vec, 5e-3)
    # the captured graph replays the same iteration
    cap = S.refine.BatchRefiner([make(k) for k in range(4)]).capture()
    cap.run(iters)
    torch.cuda.synchronize()
    # (not bit-equal: the fp32 / fp64 atomics of the reductions land in another order, and AdamW's g / sqrt(v) amplifies that)
    assert parity_ok("graph_loss", cap.loss, bat.loss, 1e-4) and parity_ok("graph_shapecode", cap.shapecode, bat.shapecode, 2e-2, outliers=ADAM_OUTLIERS)
    with pytest.raises(ValueError):
        cap.run(1)            # the jitter tables hold max_iters rows


@pytest.mark.parametrize("blocks,B,n,S_", [((3, 1), 1, 128, 16), ((3, 1), 4, 64, 8), ((5, 5), 2, 32, 8), ((2, 1), 1, 37, 5)])
def test_decoder_fp32_on_tensor_cores_vs_oracle(blocks, B, n, S_):
    """SNB_PREC_FP32_TC (fp32 mode with frozen weights: two fp16 parts per MMA operand, three tcgen05 MMAs per product) against the fp32
    oracle at the fp32 tolerance -- outputs, d xyz, d viewdir and the latent gradients -- with per-row upstream gradients spread over 12
    orders of magnitude (compositing weights do that) and a few all-zero rows, and beside the FFMA back end's own errors."""
    S = snb()
    sd = oracle.init_codenerf_state(shape_blocks=blocks[0], texture_blocks=blocks[1], seed=blocks[0] + 20)
    xyz, vd, shp, tex, up_s, up_c = _decoder_case(None, sd, None, B, n, S_, seed=blocks[0] * 10 + B + 3)
    g = torch.Generator().manual_seed(9)
    row_mag = 10.0 ** (torch.rand(B * n, S_, 1, generator=g) * 12 - 9)
    row_mag[::7] = 0.0
    up_s, up_c = up_s * row_mag, up_c * row_mag

    def run_oracle(dt):
        sdd = {k: v.to(dt) for k, v in sd.items()}
        ins = [t.detach().clone().to(dt).requires_grad_() for t in (xyz, vd, shp, tex)]
        sig, rgbs = oracle.codenerf_decoder(sdd, *ins)
        ((sig * up_s.to(dt)).sum() + (rgbs * up_c.to(dt)).sum()).backward()
        return [sig.detach(), rgbs.detach()] + [t.grad for t in ins]
    ref, truth = run_oracle(torch.float32), run_oracle(torch.float64)
    m = model_from_state(S.CodeNeRF, sd, shape_blocks=blocks[0], texture_blocks=blocks[1])
    m.precision = "fp32"
    m.requires_grad_(False)

    def run_gpu(tensor_cores):
        old = S.ops.FP32_TENSOR_CORES
        S.ops.FP32_TENSOR_CORES = tensor_cores
        try:
            gin = [t.detach().clone().to(DEV).requires_grad_() for t in (xyz, vd, shp, tex)]
            before = S._lib.load().snb_launch_count()
            sig2, rgbs2 = m(*gin)
            ((sig2 * up_s.to(DEV)).sum() + (rgbs2 * up_c.to(DEV)).sum()).backward()
            return [sig2.detach(), rgbs2.detach()] + [t.grad for t in gin], S._lib.load().snb_launch_count() - before
        finally:
            S.ops.FP32_TENSOR_CORES = old
    got, launches_tc = run_gpu(True)
    simt, launches_simt = run_gpu(False)
    assert launches_tc < launches_simt            # the tensor-core path is 2 decoder kernels + the latent layers, not one SGEMM per layer
    for name, a, s_, r, t in zip(("sigma", "rgb", "g_xyz", "g_viewdir", "g_shape", "g_texture"), got, simt, ref, truth):
        assert close_vs_truth(a, r, t, name="tc_" + name)[0], (name, close_vs_truth(a, r, t))
        parity_ok("simt_" + name, s_, r, 1.0)     # ledger only: the FFMA back end's error on the same case


def test_batched_render_fp32_tensor_cores_vs_per_object_and_oracle():
    """The batched box render with the decoder in SNB_PREC_FP32_TC arithmetic (model.precision = 'fp32', frozen weights): against the
    per-object fused render of the same precision (same per-row arithmetic: hit rays bit-identical) and against the fp32 / fp64 CPU
    oracle at the fp32 tolerance -- render, loss and the pose / code gradients."""
    S = snb()
    if not S.ops.FP32_TENSOR_CORES:
        pytest.skip("SNB_FP32_SIMT=1: the per-object render runs on the FFMA kernels, nothing to compare bit for bit")
    n_obj, im, S_ = 3, 24, 32
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=62)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = "fp32"
    m.requires_grad_(False)
    R = S.renderer.NeRFRenderer(n_samples=S_)
    objs = [oracle.synthetic_object(230 + 7 * i, im_sz=im) for i in range(n_obj)]
    lat = [oracle.synthetic_latents(230 + 7 * i, 1) for i in range(n_obj)]
    n = im * im
    jit = torch.rand(n_obj, n, S_, generator=torch.Generator().manual_seed(62))
    per = []
    for i, o in enumerate(objs):
        cam = o["cam_pose"].to(DEV).requires_grad_()
        shp, tex = lat[i][0].to(DEV).requires_grad_(), lat[i][1].to(DEV).requires_grad_()
        with forced_rand_like(jit[i]):
            rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, o["img"], o["mask_occ"], cam, o["wlh"], o["K"].to(DEV), o["roi"], shp, tex, im_sz=im)
        S.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0].backward()
        per.append((rgb.detach(), dep.detach(), acc.detach(), cam.grad, shp.grad, tex.grad))
    cams = torch.stack([o["cam_pose"] for o in objs]).to(DEV).requires_grad_()
    shps = torch.cat([l[0] for l in lat]).to(DEV).requires_grad_()
    texs = torch.cat([l[1] for l in lat]).to(DEV).requires_grad_()
    before = S._lib.load().snb_launch_count()
    rgb, dep, acc, tgt, occ = R.render_rays_batch(m, DEV, [o["img"] for o in objs], [o["mask_occ"] for o in objs], cams,
                                                  [o["wlh"] for o in objs], torch.stack([o["K"] for o in objs]), [o["roi"] for o in objs],
                                                  shps, texs, im_sz=im, jitter=jit.to(DEV))
    losses, _ = S.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)
    losses.sum().backward()
    assert S._lib.load().snb_launch_count() - before <= 30          # one launch set for the three objects (per object: ~24 each)
    for i, o in enumerate(objs):
        ro, vd = oracle.get_rays(o["K"], o["cam_pose"], o["roi"], uv_steps=[im, im])
        diag, half = oracle.box_constants(o["wlh"])
        hb = torch.from_numpy(half)
        hit = oracle.ray_box_intersection(ro / (diag / 2), vd, -hb.expand_as(ro), hb.expand_as(ro))[2].to(DEV)
        for a, b_ in zip((rgb[i], dep[i], acc[i]), per[i][:3]):
            assert torch.equal(a[hit], b_[hit])
        assert parity_ok("obj%d_g_shape_vs_per_object" % i, shps.grad[i], per[i][4][0], 1e-4)
        assert parity_ok("obj%d_g_pose_vs_per_object" % i, cams.grad[i], per[i][3], 1e-3)
        res = {}
        for dt in (torch.float32, torch.float64):
            sdd = {k: v.to(dt) for k, v in sd.items()}
            cam_o = o["cam_pose"].to(dt).clone().requires_grad_()
            s_o, t_o = lat[i][0].to(dt).clone().requires_grad_(), lat[i][1].to(dt).clone().requires_grad_()
            r_o = oracle.render_rays_box(sdd, o["K"].to(dt), cam_o, o["wlh"], o["roi"], im, S_, s_o, t_o, jit[i].to(dt))
            l_o = oracle.refine_losses(r_o[0], r_o[2], o["img"].reshape(-1, 3).to(dt), o["mask_occ"].reshape(-1, 1).to(dt))[0]
            l_o.backward()
            res[dt] = (r_o[0].detach(), r_o[1].detach(), l_o.detach(), cam_o.grad, s_o.grad[0], t_o.grad[0])
        got = (rgb[i], dep[i], losses[i], cams.grad[i], shps.grad[i], texs.grad[i])
        for name, a, r32, r64 in zip(("rgb", "depth", "loss", "g_pose", "g_shape", "g_texture"), got, res[torch.float32], res[torch.float64]):
            assert close_vs_truth(a, r32, r64, name="obj%d_%s_vs_oracle" % (i, name))[0], (i, name, close_vs_truth(a, r32, r64))


def test_fp32_tensor_core_mode_steps_aside_for_weights_outside_fp16_range():
    """The split-precision kernels hold 256 * w in fp16 pairs: a weight set with |w| >= 255 must run on the FFMA kernels instead (checked
    once per weight version on the device) -- same results as ever, no inf."""
    S = snb()
    sd = oracle.init_codenerf_state(shape_blocks=2, texture_blocks=1, seed=31)
    sd["shape_layer_1.0.weight"] = sd["shape_layer_1.0.weight"].clone()
    sd["shape_layer_1.0.weight"][3, 5] = 300.0
    xyz, vd, shp, tex, _, _ = _decoder_case(None, sd, None, 1, 64, 8, seed=12)
    sig, rgbs = oracle.codenerf_decoder(sd, xyz, vd, shp, tex)
    m = model_from_state(S.CodeNeRF, sd, shape_blocks=2, texture_blocks=1)
    m.precision = "fp32"
    m.requires_grad_(False)
    h = m._handle(torch.device(DEV, torch.cuda.current_device()))
    assert h.tc_ok and not h.weights_in_fp16_range(m._weights())
    sig2, rgbs2 = m(xyz.to(DEV), vd.to(DEV), shp.to(DEV), tex.to(DEV))
    assert bool(torch.isfinite(sig2).all()) and bool(torch.isfinite(rgbs2).all())
    assert parity_ok("sigma", sig2, sig, TOL) and parity_ok("rgb", rgbs2, rgbs, TOL)
    with torch.no_grad():
        m.get_parameter("shape_layer_1.0.weight")[3, 5] = 0.01      # an in-place update bumps the version: re-checked, back on the tensor cores
    assert h.weights_in_fp16_range(m._weights())


# ------------------------------------------------------------------------------------------- counter-based jitter
_M32 = np.uint64(0xFFFFFFFF)


def _philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11; Random123), vectorised over numpy uint64 arrays that hold 32-bit words."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) for c in ctr)
    k0, k1 = (np.asarray(k, dtype=np.uint64) for k in key)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c0, np.uint64(0xCD9E8D57) * c2      # < 2^64: exact
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & _M32, (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def _jitter_reference(seed, ray_ids, n_samples):
    """u[r][k] = word k % 4 of Philox4x32-10(counter (id low, id high, k / 4, 0), key (seed low, seed high)), as (x >> 8) * 2^-24."""
    ids = np.asarray(ray_ids, dtype=np.uint64)[:, None]
    k = np.arange(n_samples, dtype=np.uint64)[None, :]
    seed = np.uint64(seed)
    words = np.stack(np.broadcast_arrays(*_philox4x32_10((ids & _M32, ids >> np.uint64(32), k // np.uint64(4), np.uint64(0)),
                                                         (seed & _M32, seed >> np.uint64(32)))), -1)
    x = np.take_along_axis(words, np.broadcast_to((k % np.uint64(4)).astype(np.int64)[..., None], words.shape[:2] + (1,)), -1)[..., 0]
    return torch.from_numpy(((x >> np.uint64(8)).astype(np.float64) * 2.0 ** -24).astype(np.float32))


@pytest.mark.parametrize("S_", [1, 3, 4, 7, 64])
def test_jitter_fill_is_philox4x32_10_bit_for_bit(S_):
    """ops.jitter_fill (snb_jitter_fill, the ray-sharded modes' stratified jitter) against a Python Philox4x32-10 that reproduces the
    Random123 known-answer vectors: every value bit for bit, seeds and ray ids past 2^32, and shards given by ray ids whose union is the
    full draw."""
    hexw = lambda ws: ["%08x" % int(w) for w in ws]   # noqa: E731
    assert hexw(_philox4x32_10([0] * 4, [0, 0])) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    assert hexw(_philox4x32_10([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2)) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert hexw(_philox4x32_10([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0])) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]
    S = snb()
    n = 777
    for seed in (0, 20240611, (1 << 32) + 5, (1 << 64) - 3):
        full = S.ops.jitter_fill(seed, n, S_, DEV)
        assert full.shape == (n, S_) and torch.equal(full.cpu(), _jitter_reference(seed, np.arange(n), S_))
        ids = torch.arange(n, dtype=torch.int64) + (1 << 32) - 300          # both sides of 2^32
        ids[-5:] = torch.tensor([(1 << 40) + 1, (1 << 48) + 77, (1 << 62) + 3, (1 << 63) - 1, 12345])
        big = S.ops.jitter_fill(seed, 0, S_, DEV, ray_ids=ids.to(DEV))
        assert torch.equal(big.cpu(), _jitter_reference(seed, ids.numpy(), S_))
        assert float(big.min()) >= 0.0 and float(big.max()) < 1.0
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(S_))
        union = torch.full((n, S_), -1.0)
        for shard in (perm[:100], perm[100:101], perm[101:]):
            union[shard] = S.ops.jitter_fill(seed, 0, S_, DEV, ray_ids=ids[shard].to(DEV)).cpu()
        assert torch.equal(union, big.cpu())
