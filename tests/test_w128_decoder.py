"""The CodeNeRF-family decoder at hidden width W = 128 (AutoRFMix()'s class defaults: 5 + 5 blocks, W = latent_dim = 128) on the one-tile
tcgen05 kernels, in bf16 and in split precision (fp32 mode, frozen weights): the size queries (no device needed), and on the GPU the
decoder, the debug dump, the per-object and batched renders, the graphed batch step and the batched refiner against the oracle."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import close_vs_truth, parity, parity_ok, rel_err
from oracle import oracle

TOL = 2e-2
AUTORFMIX = (5, 5, 128, 128)           # shape_blocks, texture_blocks, W, latent_dim: AutoRFMix() class defaults
CODENERF_W128 = (2, 1, 128, 256)       # CodeNeRF(2, 1, W=128, latent_dim=256): latent_dim != W
DEV = "cuda"


def _handle(blocks_s, blocks_t, W, D):
    from supnerf_b200 import ops
    return ops.DecoderHandle(0, blocks_s, blocks_t, W, D, 10, 4)


def _lib():
    from supnerf_b200 import _lib
    return _lib.load()


# ------------------------------------------------------------------------------------------------ size queries (CPU)
def test_w256_sizes_unchanged():
    lib = _lib()
    for arch, ws, packed in (((3, 1, 256, 256), 235536640, 10083328), ((5, 5, 256, 256), 437846272, 13633536)):
        h = _handle(*arch)
        assert h.tc_ok
        for p in (1, 3):
            assert lib.snb_mlp_workspace_bytes(h.h, 2 ** 20, 16, p) == ws, (arch, p)
        assert lib.snb_packed_bytes(h.h) == packed, arch


@pytest.mark.parametrize("arch", [AUTORFMIX, CODENERF_W128])
def test_w128_on_the_tensor_cores(arch):
    lib = _lib()
    h = _handle(*arch)
    assert h.tc_ok
    ws = lib.snb_mlp_workspace_bytes(h.h, 2 ** 20, 16, 1)
    assert lib.snb_mlp_workspace_bytes(h.h, 2 ** 20, 16, 3) == ws
    assert ws < lib.snb_mlp_workspace_bytes(_handle(5, 5, 256, 256).h, 2 ** 20, 16, 1)
    # per latent slot and object W floats each of zlat and the effective biases and 32 bytes per unit of their bias-stage images;
    # per 128-row tile and layer W / 32 mask words of 128 rows
    slots, tiles = arch[0] + arch[1], 2 ** 20 // 128
    assert ws == 256 + slots * 16 * arch[2] * (4 + 4 + 32) + tiles * (slots + 3) * (arch[2] // 32) * 128 * 4
    assert lib.snb_packed_bytes(h.h) > 16


@pytest.mark.parametrize("W", [64, 192])
def test_other_widths_stay_off_the_tensor_cores(W):
    assert not _handle(2, 1, W, W).tc_ok


# ------------------------------------------------------------------------------------------------ GPU
def _snb():
    import supnerf_b200
    return supnerf_b200


def _model(arch, sd):
    S = _snb()
    if arch == AUTORFMIX:
        m = S.AutoRFMix()
    else:
        m = S.CodeNeRF(shape_blocks=arch[0], texture_blocks=arch[1], W=arch[2], latent_dim=arch[3])
    m.load_state_dict({k: v.detach().clone() for k, v in sd.items()})
    return m.to(DEV)


def _state(arch, seed):
    return oracle.init_codenerf_state(shape_blocks=arch[0], texture_blocks=arch[1], W=arch[2], latent_dim=arch[3], seed=seed)


def _case(arch, B, n, S_, seed):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(B * n, S_, 3, generator=g) - 0.5) * 1.6
    vd = torch.nn.functional.normalize(torch.randn(B * n, 1, 3, generator=g), dim=-1).repeat(1, S_, 1)
    shp, tex = oracle.synthetic_latents(seed, B, arch[3])
    up_s, up_c = torch.randn(B * n, S_, 1, generator=g), torch.randn(B * n, S_, 3, generator=g)
    return xyz, vd, shp, tex, up_s, up_c


# (arch, B, n, S): 256 and 128 rows per object, and one object of 150 rows (padded to two 128-row tiles)
CASES = [(AUTORFMIX, 2, 16, 16), (AUTORFMIX, 3, 8, 16), (CODENERF_W128, 1, 10, 15), (CODENERF_W128, 2, 32, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("arch,B,n,S_", CASES)
def test_w128_bf16_decoder_fwd_bwd_vs_oracle(arch, B, n, S_):
    """As test_gpu_bf16.py's test_tc_decoder_fwd_bwd_vs_oracle: against the bf16 emulation (its own distance to the fp32 oracle as
    the floor) and, under a smooth upstream gradient, the latent gradients against the fp32 oracle at 2e-2."""
    sd = _state(arch, seed=arch[0] + 40)
    xyz, vd, shp, tex, up_s, up_c = _case(arch, B, n, S_, arch[0] * 7 + B + 40)
    ins = [t.clone().requires_grad_() for t in (xyz, vd, shp, tex)]
    sig, rgbs = oracle.codenerf_decoder(sd, *ins)
    ((sig * up_s).sum() + (rgbs * up_c).sum()).backward()
    ine = [t.clone().requires_grad_() for t in (xyz, vd, shp, tex)]
    sig_e, rgbs_e = oracle.codenerf_decoder_bf16(sd, *ine)
    ((sig_e * up_s).sum() + (rgbs_e * up_c).sum()).backward()
    m = _model(arch, sd)
    m.precision = "bf16"
    m.requires_grad_(False)
    gin = [t.to(DEV).requires_grad_() for t in (xyz, vd, shp, tex)]
    sig2, rgbs2 = m(*gin)
    assert parity_ok("sig2", sig2, sig, TOL) and parity_ok("rgbs2", rgbs2, rgbs, TOL)
    assert parity_ok("sig2_vs_emulation", sig2, sig_e, 5e-3) and parity_ok("rgbs2_vs_emulation", rgbs2, rgbs_e, 5e-3)
    ((sig2 * up_s.to(DEV)).sum() + (rgbs2 * up_c.to(DEV)).sum()).backward()
    names = ("xyz", "viewdir", "shape", "texture")
    for a, b, c, n_ in zip(gin, ins, ine, names):
        floor = rel_err(c.grad, b.grad)
        parity("g_%s_vs_bf16_emulation" % n_, a.grad, c.grad, TOL, floor=floor, floor_slack=1.0)
        parity("g_%s_vs_fp32_oracle" % n_, a.grad, b.grad, TOL, floor=floor)
    us, uc = torch.tensor(0.7), torch.tensor([0.3, -0.5, 0.9])
    ins_s = [t.clone().requires_grad_() for t in (xyz, vd, shp, tex)]
    sig_s, rgbs_s = oracle.codenerf_decoder(sd, *ins_s)
    ((sig_s * us).sum() + (rgbs_s * uc).sum()).backward()
    gin_s = [t.to(DEV).requires_grad_() for t in (xyz, vd, shp, tex)]
    sig4, rgbs4 = m(*gin_s)
    ((sig4 * us.to(DEV)).sum() + (rgbs4 * uc.to(DEV)).sum()).backward()
    for a, b, n_ in zip(gin_s[2:], ins_s[2:], names[2:]):
        parity("smooth_upstream_g_%s" % n_, a.grad, b.grad, TOL)
    # latents only (the backward program without d xyz / d viewdir): the same latent gradients
    gin2 = [t.to(DEV) for t in (xyz, vd)] + [t.to(DEV).requires_grad_() for t in (shp, tex)]
    sig3, rgbs3 = m(*gin2)
    ((sig3 * up_s.to(DEV)).sum() + (rgbs3 * up_c.to(DEV)).sum()).backward()
    assert parity_ok("latents_only_g_shape", gin2[2].grad, gin[2].grad, 1e-4)
    assert parity_ok("latents_only_g_texture", gin2[3].grad, gin[3].grad, 1e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("arch,B,n,S_", [c for c in CASES if (c[2] * c[3]) % 128 == 0])
def test_w128_split_precision_decoder_vs_oracle(arch, B, n, S_):
    """fp32 mode with frozen weights (SNB_PREC_FP32_TC) against the fp32 / fp64 oracle at 1e-5, with per-row upstream gradients spread
    over 12 orders of magnitude and some all-zero rows; on fewer launches than the FFMA back end; latents-only backward as the full one."""
    S = _snb()
    if not S.ops.FP32_TENSOR_CORES:
        pytest.skip("SNB_FP32_SIMT=1: fp32 mode runs on the FFMA kernels")
    sd = _state(arch, seed=arch[0] + 50)
    xyz, vd, shp, tex, up_s, up_c = _case(arch, B, n, S_, arch[0] * 11 + B + 50)
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
    m = _model(arch, sd)
    m.precision = "fp32"
    m.requires_grad_(False)

    def run_gpu(tensor_cores, latents_only=False):
        old = S.ops.FP32_TENSOR_CORES
        S.ops.FP32_TENSOR_CORES = tensor_cores
        try:
            gin = [t.detach().clone().to(DEV).requires_grad_(not latents_only or i >= 2) for i, t in enumerate((xyz, vd, shp, tex))]
            before = S._lib.load().snb_launch_count()
            sig2, rgbs2 = m(*gin)
            ((sig2 * up_s.to(DEV)).sum() + (rgbs2 * up_c.to(DEV)).sum()).backward()
            return [sig2.detach(), rgbs2.detach()] + [t.grad for t in gin], S._lib.load().snb_launch_count() - before
        finally:
            S.ops.FP32_TENSOR_CORES = old
    got, launches_tc = run_gpu(True)
    _, launches_simt = run_gpu(False)
    assert launches_tc < launches_simt
    for name, a, r, t in zip(("sigma", "rgb", "g_xyz", "g_viewdir", "g_shape", "g_texture"), got, ref, truth):
        assert close_vs_truth(a, r, t, name="w128_tc_" + name)[0], (name, close_vs_truth(a, r, t))
    lat, _ = run_gpu(True, latents_only=True)
    assert parity_ok("latents_only_g_shape", lat[4], got[4], 1e-5) and parity_ok("latents_only_g_texture", lat[5], got[5], 1e-5)


@pytest.mark.gpu
def test_w128_forward_layer_by_layer():
    """Every layer's output from the debug dump ([steps][rows][256], the first W or W / 2 columns written) against the oracle."""
    S = _snb()
    sd = _state(AUTORFMIX, seed=6)
    xyz, vd, shp, tex, _, _ = _case(AUTORFMIX, 2, 16, 16, 6)
    with torch.no_grad():
        sig, rgbs, acts = oracle.codenerf_decoder(sd, xyz, vd, shp, tex, return_acts=True)
    m = _model(AUTORFMIX, sd)
    m.precision = "bf16"
    m.requires_grad_(False)
    M = xyz.shape[0] * xyz.shape[1]
    dbg = torch.full((len(acts), M, 256), 1234.0, device=DEV)
    lib = S._lib.load()
    hnd = m._handle(dbg.device).h
    lib.snb_tc_set_debug(hnd, ctypes.c_void_p(dbg.data_ptr()))
    try:
        with torch.no_grad():
            sig2, rgbs2 = m(xyz.to(DEV), vd.to(DEV), shp.to(DEV), tex.to(DEV))
        torch.cuda.synchronize()
    finally:
        lib.snb_tc_set_debug(hnd, None)
    for i, a in enumerate(acts):
        w = a.shape[-1]
        parity("layer_%d_activations" % i, dbg[i, :, :w], a.reshape(M, w), TOL)
        assert bool((dbg[i, :, w:] == 1234.0).all())          # nothing beyond the layer's width
    assert parity_ok("sig2", sig2, sig, TOL) and parity_ok("rgbs2", rgbs2, rgbs, TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_w128_decoder_records_tensor_core_kernel_events(prec):
    """Kernel-timing events are recorded by the tcgen05 back ends only: W = 128 records them in both precisions, the FFMA back end
    (fp32 mode forced to SIMT) records none."""
    S = _snb()
    sd = _state(AUTORFMIX, seed=7)
    xyz, vd, shp, tex, _, _ = _case(AUTORFMIX, 1, 32, 16, 7)
    m = _model(AUTORFMIX, sd)
    m.precision = prec
    m.requires_grad_(False)
    lib = S._lib.load()
    buf = (ctypes.c_float * 16)()

    def events(tensor_cores):
        old = S.ops.FP32_TENSOR_CORES
        S.ops.FP32_TENSOR_CORES = tensor_cores
        try:
            gin = [t.to(DEV).requires_grad_() for t in (xyz, vd, shp, tex)]
            hnd = m._handle(gin[0].device).h
            lib.snb_kernel_timing_enable(hnd, 1)
            sig, rgbs = m(*gin)
            (sig.sum() + rgbs.sum()).backward()
            torch.cuda.synchronize()
            n = lib.snb_kernel_timing_read(hnd, 0, buf, 16), lib.snb_kernel_timing_read(hnd, 1, buf, 16)
            lib.snb_kernel_timing_enable(hnd, 0)
            return n
        finally:
            S.ops.FP32_TENSOR_CORES = old
    n_fwd, n_bwd = events(True)
    assert n_fwd >= 1 and n_bwd >= 1
    if prec == "fp32":
        assert events(False) == (0, 0)


@pytest.mark.gpu
def test_autorfmix_defaults_per_object_and_batched_render():
    """AutoRFMix() with its class defaults through the per-object fused render and the batched launch set, bf16 and (frozen weights)
    split precision.  Half of one object's occupancy rows and all of another's are zero, so the batched backward has dead super tiles
    to skip.  Batched vs per-object: hit rays bit-identical, code gradients within 1e-4; against the fp32 CPU oracle within each mode's
    budget."""
    S = _snb()
    if not S.ops.FP32_TENSOR_CORES:
        pytest.skip("SNB_FP32_SIMT=1: the per-object fp32 render runs on the FFMA kernels, nothing to compare bit for bit")
    n_obj, im, S_ = 3, 16, 32
    sd = _state(AUTORFMIX, seed=78)
    objs = [oracle.synthetic_object(270 + 7 * i, im_sz=im) for i in range(n_obj)]
    for o in objs:
        o["mask_occ"] = o["mask_occ"].clone()
    objs[0]["mask_occ"][: im // 2] = 0
    objs[2]["mask_occ"][:] = 0
    lat = [oracle.synthetic_latents(270 + 7 * i, 1, AUTORFMIX[3]) for i in range(n_obj)]
    n = im * im
    jit = torch.rand(n_obj, n, S_, generator=torch.Generator().manual_seed(78))
    R = S.renderer.NeRFRenderer(n_samples=S_)
    from test_gpu_parity import forced_rand_like
    for prec, tol in (("bf16", TOL), ("fp32", 1e-5)):
        m = _model(AUTORFMIX, sd)
        m.precision = prec
        m.requires_grad_(False)
        per = []
        for i, o in enumerate(objs):
            cam = o["cam_pose"].to(DEV).requires_grad_()
            shp, tex = lat[i][0].to(DEV).requires_grad_(), lat[i][1].to(DEV).requires_grad_()
            with forced_rand_like(jit[i]):
                rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, o["img"], o["mask_occ"], cam, o["wlh"], o["K"].to(DEV), o["roi"], shp, tex,
                                                        im_sz=im)
            S.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0].backward()
            per.append((rgb.detach(), dep.detach(), cam.grad, shp.grad, tex.grad))
        cams = torch.stack([o["cam_pose"] for o in objs]).to(DEV).requires_grad_()
        shps = torch.cat([l[0] for l in lat]).to(DEV).requires_grad_()
        texs = torch.cat([l[1] for l in lat]).to(DEV).requires_grad_()
        rgb, dep, acc, tgt, occ = R.render_rays_batch(m, DEV, [o["img"] for o in objs], [o["mask_occ"] for o in objs], cams,
                                                      [o["wlh"] for o in objs], torch.stack([o["K"] for o in objs]), [o["roi"] for o in objs],
                                                      shps, texs, im_sz=im, jitter=jit.to(DEV))
        S.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)[0].sum().backward()
        for i, o in enumerate(objs):
            ro, vd = oracle.get_rays(o["K"], o["cam_pose"], o["roi"], uv_steps=[im, im])
            diag, half = oracle.box_constants(o["wlh"])
            hb = torch.from_numpy(half)
            hit = oracle.ray_box_intersection(ro / (diag / 2), vd, -hb.expand_as(ro), hb.expand_as(ro))[2].to(DEV)
            assert bool(hit.any())
            assert torch.equal(rgb[i][hit], per[i][0][hit]) and torch.equal(dep[i][hit], per[i][1][hit])
            parity("%s_obj%d_g_shape_vs_per_object" % (prec, i), shps.grad[i], per[i][3][0], 1e-4)
            parity("%s_obj%d_g_texture_vs_per_object" % (prec, i), texs.grad[i], per[i][4][0], 1e-4)
            cam_o = o["cam_pose"].clone().requires_grad_()
            s_o, t_o = lat[i][0].clone().requires_grad_(), lat[i][1].clone().requires_grad_()
            rgb_o, dep_o, acc_o, _ = oracle.render_rays_box(sd, o["K"], cam_o, o["wlh"], o["roi"], im, S_, s_o, t_o, jit[i])
            oracle.refine_losses(rgb_o, acc_o, o["img"].reshape(-1, 3), o["mask_occ"].reshape(-1, 1))[0].backward()
            parity("%s_obj%d_rgb_vs_oracle" % (prec, i), rgb[i], rgb_o, tol)
            parity("%s_obj%d_depth_vs_oracle" % (prec, i), dep[i], dep_o, tol)
            if i == 2:          # no occupied pixel: the object's loss does not depend on its codes
                assert float(shps.grad[i].abs().max()) == 0.0 and float(texs.grad[i].abs().max()) == 0.0
            else:
                parity("%s_obj%d_g_shape_vs_oracle" % (prec, i), shps.grad[i], s_o.grad[0], tol if prec == "bf16" else 1e-4)


@pytest.mark.gpu
def test_autorfmix_defaults_graphed_batch_step_equals_the_call_by_call_step():
    """renderer.GraphedBatchStep with AutoRFMix() defaults: one replay against the same step issued call by call, same jitter."""
    S = _snb()
    n_obj, im, S_ = 3, 16, 32
    sd = _state(AUTORFMIX, seed=92)
    m = _model(AUTORFMIX, sd)
    m.precision = "bf16"
    m.requires_grad_(False)
    R = S.renderer.NeRFRenderer(n_samples=S_)
    objs = [oracle.synthetic_object(310 + 7 * i, im_sz=im) for i in range(n_obj)]
    lat = [oracle.synthetic_latents(310 + 7 * i, 1, AUTORFMIX[3]) for i in range(n_obj)]
    pin = lambda t: t.contiguous().float().pin_memory()   # noqa: E731
    h_img, h_mask = pin(torch.stack([o["img"] for o in objs])), pin(torch.stack([o["mask_occ"] for o in objs]))
    h_cam, h_K = pin(torch.stack([o["cam_pose"] for o in objs])), pin(torch.stack([o["K"] for o in objs]))
    h_shp, h_tex = pin(torch.cat([l[0] for l in lat])), pin(torch.cat([l[1] for l in lat]))
    wlhs, rois = [o["wlh"] for o in objs], [o["roi"] for o in objs]
    jit = torch.rand(n_obj, im * im, S_, generator=torch.Generator().manual_seed(92)).to(DEV)
    step = S.renderer.GraphedBatchStep(R, m, DEV, h_img, h_mask, h_cam, wlhs, h_K, rois, h_shp, h_tex, im_sz=im, jitter=jit)
    got = step.run()
    torch.cuda.synchronize()
    got = got.clone()
    cam, shp, tex = [t.to(DEV).requires_grad_() for t in (h_cam, h_shp, h_tex)]
    rgb, dep, acc, tgt, occ = R.render_rays_batch(m, DEV, h_img, h_mask, cam, wlhs, h_K, rois, shp, tex, im_sz=im, jitter=jit)
    loss, parts = S.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)
    loss.backward(gradient=torch.ones(n_obj, device=DEV))
    ref = torch.cat([parts[:, :1], cam.grad.reshape(n_obj, 12), shp.grad, tex.grad], 1).cpu()
    assert got.shape == (n_obj, 1 + 12 + 2 * AUTORFMIX[3])
    parity("loss", got[:, 0], ref[:, 0], 1e-6)
    parity("g_pose", got[:, 1:13], ref[:, 1:13], 1e-4)
    parity("g_codes", got[:, 13:], ref[:, 13:], 1e-5)
    assert float(got[:, 0].abs().min()) > 0


@pytest.mark.gpu
def test_autorfmix_defaults_batch_refiner_losses_go_down():
    """refine.BatchRefiner over 2 objects with AutoRFMix() defaults in bf16: finite losses that decrease over a few iterations."""
    S = _snb()
    import tools.refine_bench as rb
    sd = _state(AUTORFMIX, seed=54)
    m = _model(AUTORFMIX, sd)
    m.precision = "bf16"
    m.requires_grad_(False)
    iters = 8

    def make(k):
        seed = 90 + k
        obj = oracle.synthetic_object(seed, im_sz=32)
        shp0, tex0 = oracle.synthetic_latents(seed, 1, AUTORFMIX[3])
        c2o = obj["cam_pose"]
        R_obj = c2o[:, :3].t().contiguous()
        t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
        torch.manual_seed(seed)
        return S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                      shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, n_samples=64, im_sz=32, max_iters=iters)
    bat = S.refine.BatchRefiner([make(k) for k in range(2)])
    losses = []
    for _ in range(iters):
        losses.append(bat.run(1)[:, 0].clone())
    losses = torch.stack(losses).cpu()           # (iters, objects)
    print("losses per iteration:", losses.tolist())
    assert bool(torch.isfinite(losses).all())
    assert bool((losses[-1] < losses[0]).all())


@pytest.mark.gpu
def test_w128_training_bf16_raises_fp32_gives_weight_grads():
    """Weight gradients at W = 128: bf16 still refuses (they need the two-tile kernels); fp32 computes them on the FFMA back end."""
    sd = _state(AUTORFMIX, seed=8)
    xyz, vd, shp, tex, up_s, up_c = _case(AUTORFMIX, 1, 8, 16, 8)
    m = _model(AUTORFMIX, sd)
    m.precision = "bf16"
    with pytest.raises(RuntimeError):
        sig, rgbs = m(xyz.to(DEV), vd.to(DEV), shp.to(DEV), tex.to(DEV))
        (sig.sum() + rgbs.sum()).backward()
    m = _model(AUTORFMIX, sd)
    m.precision = "fp32"
    sig, rgbs = m(xyz.to(DEV), vd.to(DEV), shp.to(DEV), tex.to(DEV))
    ((sig * up_s.to(DEV)).sum() + (rgbs * up_c.to(DEV)).sum()).backward()

    def run_oracle(dt):
        sdd = {k: v.detach().clone().to(dt).requires_grad_() for k, v in sd.items()}
        s_, c_ = oracle.codenerf_decoder(sdd, *[t.to(dt) for t in (xyz, vd, shp, tex)])
        ((s_ * up_s.to(dt)).sum() + (c_ * up_c.to(dt)).sum()).backward()
        return sdd
    ref, truth = run_oracle(torch.float32), run_oracle(torch.float64)
    for k, p in m.named_parameters():
        assert p.grad is not None, k
        assert close_vs_truth(p.grad, ref[k].grad, truth[k].grad, name="fp32_train_gw_" + k)[0], k
