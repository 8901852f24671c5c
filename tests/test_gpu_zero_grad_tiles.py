"""The batched render's decoder backward runs only the 256-row super tiles whose upstream gradient is not exactly zero
(csrc/render_batch.cu: live flags + list; the tcgen05 backward kernels walk the list).  Rays the refine loss gives no weight
(occ == 0) make whole super tiles dead.  Their rows' d xyz / d viewdir are not written this call, so the rays backward must not
read them: stale or poisoned scratch would leak into the pose gradient.  Every case: against the per-object render of the same
library (tolerances of test_batched_render_equals_per_object_render) and, in bf16, against the fp32 CPU oracle."""
import ctypes

import pytest
import torch

from conftest import TRUTH_SLACK, close_vs_truth, parity, rel_err
from oracle import oracle
from test_gpu_parity import DEV, forced_rand_like, model_from_state, snb

pytestmark = pytest.mark.gpu
TOL = 2e-2


def _setup(prec, n_obj, im, S_, seed):
    S = snb()
    if prec == "fp32" and not S.ops.FP32_TENSOR_CORES:
        pytest.skip("SNB_FP32_SIMT=1: no split-precision tensor-core decoder to test")
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=seed)
    m = model_from_state(S.SUPNeRF, sd, 3, 1, 3, 3, 256)
    m.precision = prec
    m.requires_grad_(False)
    R = S.renderer.NeRFRenderer(n_samples=S_)
    objs = [oracle.synthetic_object(seed + 7 * i, im_sz=im) for i in range(n_obj)]
    lat = [oracle.synthetic_latents(seed + 7 * i, 1) for i in range(n_obj)]
    jit = torch.rand(n_obj, im * im, S_, generator=torch.Generator().manual_seed(seed))
    return S, sd, m, R, objs, lat, jit


def _all_live(mask):
    return torch.where(mask == 0, torch.ones_like(mask), mask)       # occ = +-1 everywhere: every super tile live


def _band(mask, r0, r1):
    out = _all_live(mask).clone()
    out[r0:r1] = 0.0        # a band of whole pixel rows: consecutive hit rays, so whole super tiles get no gradient
    return out


def _batched(S, m, R, objs, lat, jit, masks, im):
    cams = torch.stack([o["cam_pose"] for o in objs]).to(DEV).requires_grad_()
    shps = torch.cat([l[0] for l in lat]).to(DEV).requires_grad_()
    texs = torch.cat([l[1] for l in lat]).to(DEV).requires_grad_()
    rgb, dep, acc, tgt, occ = R.render_rays_batch(m, DEV, [o["img"] for o in objs], masks, cams, [o["wlh"] for o in objs],
                                                  torch.stack([o["K"] for o in objs]), [o["roi"] for o in objs], shps, texs, im_sz=im,
                                                  jitter=jit.to(DEV))
    losses, _ = S.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)
    losses.sum().backward()
    torch.cuda.synchronize()
    return cams.grad, shps.grad, texs.grad


class _AbiBatch:
    """The batched render through the C ABI with a workspace and a scratch buffer the test owns: forward, the refine losses'
    upstream gradients (torch autograd on the outputs), then snb_render_batch_bwd into the given scratch."""

    def __init__(self, S, m, R, objs, lat, jit, masks, im, prec):
        self.S, self.lib, self.P = S, S._lib.load(), S._lib.ptr
        S_ = R.n_samples
        self.bt = R.make_batch(DEV, torch.stack([o["img"] for o in objs]), torch.stack(masks), [o["wlh"] for o in objs],
                               torch.stack([o["K"] for o in objs]), [o["roi"] for o in objs], im)
        self.cams = torch.stack([o["cam_pose"] for o in objs]).to(DEV)
        self.shps = torch.cat([l[0] for l in lat]).to(DEV)
        self.texs = torch.cat([l[1] for l in lat]).to(DEV)
        self.handle = m._handle(torch.device(DEV))
        flags = S.ops.SIGMA_RELU | (S.ops.BATCH_FP32_TC if prec == "fp32" else 0)
        self.handle.use_frozen(m._weights(), S.ops.PREC_FP32_TC if prec == "fp32" else S.ops.PREC["bf16"])
        b, n = self.bt.px.shape
        self.desc = S._lib.SnbBatchDesc(b, S_, n, flags, 0)
        self.scratch_bytes = self.lib.snb_render_batch_scratch_bytes(self.handle.h, ctypes.byref(self.desc))
        self.ws = torch.empty(self.lib.snb_render_batch_workspace_bytes(self.handle.h, ctypes.byref(self.desc)), dtype=torch.uint8, device=DEV)
        self.z_steps = S.renderer._z_steps_on(DEV, S_)
        self.jd = jit.to(DEV).contiguous()

    def _args(self):
        bt, P = self.bt, self.P
        return (self.handle.h, ctypes.byref(self.desc), P(bt.px), P(bt.py), P(bt.K), P(self.cams), P(bt.box), P(self.z_steps), P(self.jd),
                P(self.shps), P(self.texs))

    def backward(self, scratch):
        S, P, lib, bt = self.S, self.P, self.lib, self.bt
        b, n = bt.px.shape
        rgb, dep, acc = torch.empty(b, n, 3, device=DEV), torch.empty(b, n, device=DEV), torch.empty(b, n, device=DEV)
        st = S._lib.stream_ptr()
        S._lib.check(lib.snb_render_batch_fwd(*self._args(), P(rgb), P(dep), P(acc), None, P(self.ws), st), "snb_render_batch_fwd")
        rg, ag = rgb.clone().requires_grad_(), acc.clone().requires_grad_()
        S.losses.refine_loss_batch(rg, ag, bt.rgb_tgt, bt.occ_pixels, 0.1)[0].sum().backward()
        g_c2w = torch.empty(b, 3, 4, device=DEV)
        g_s, g_t = torch.empty_like(self.shps), torch.empty_like(self.texs)
        S._lib.check(lib.snb_render_batch_bwd(*self._args(), P(self.ws), P(rg.grad.contiguous()), None, P(ag.grad.contiguous()), P(scratch),
                                              P(g_c2w), P(g_s), P(g_t), st), "snb_render_batch_bwd")
        torch.cuda.synchronize()
        return g_c2w, g_s, g_t


def _per_object(S, m, R, o, lat_i, jit_i, mask, im):
    cam = o["cam_pose"].to(DEV).requires_grad_()
    shp, tex = lat_i[0].to(DEV).requires_grad_(), lat_i[1].to(DEV).requires_grad_()
    with forced_rand_like(jit_i):
        rgb, dep, acc, tgt, occ = R.render_rays(m, DEV, o["img"], mask, cam, o["wlh"], o["K"].to(DEV), o["roi"], shp, tex, im_sz=im)
    S.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0].backward()
    return cam.grad, shp.grad[0], tex.grad[0]


def _check_vs_per_object(name, S, m, R, objs, lat, jit, masks, im, got):
    for i, o in enumerate(objs):
        ref = _per_object(S, m, R, o, lat[i], jit[i], masks[i], im)
        parity("%s_obj%d_g_shape" % (name, i), got[1][i], ref[1], 1e-4)
        parity("%s_obj%d_g_texture" % (name, i), got[2][i], ref[2], 1e-4)
        parity("%s_obj%d_g_pose" % (name, i), got[0][i], ref[0], 1e-3)


def _check_vs_oracle(name, prec, sd, o, lat_i, jit_i, mask, im, S_, got_i, per_object_i):
    """bf16: against the fp32 oracle within the bf16 budget.  fp32 (split-precision tensor cores): close_vs_truth against the fp32
    oracle with the fp64 oracle as the truth, as test_batched_render_fp32_tensor_cores_vs_per_object_and_oracle does.  The pose
    gradient is a sum with heavy cancellation: where the split-precision arithmetic itself is further from the truth than the fp32
    oracle, it must be no further than the per-object render (same per-row arithmetic, no tiles skipped) is."""
    res = {}
    for dt in ((torch.float32,) if prec == "bf16" else (torch.float32, torch.float64)):
        sdd = {k: v.to(dt) for k, v in sd.items()}
        cam_o = o["cam_pose"].to(dt).clone().requires_grad_()
        s_o, t_o = lat_i[0].to(dt).clone().requires_grad_(), lat_i[1].to(dt).clone().requires_grad_()
        r_o = oracle.render_rays_box(sdd, o["K"].to(dt), cam_o, o["wlh"], o["roi"], im, S_, s_o, t_o, jit_i.to(dt))
        oracle.refine_losses(r_o[0], r_o[2], o["img"].reshape(-1, 3).to(dt), mask.reshape(-1, 1).to(dt))[0].backward()
        res[dt] = (cam_o.grad, s_o.grad[0], t_o.grad[0])
    for k, what in enumerate(("g_pose", "g_shape", "g_texture")):
        if prec == "bf16":
            parity("%s_%s_vs_oracle" % (name, what), got_i[k], res[torch.float32][k], TOL)
        else:
            ok = close_vs_truth(got_i[k], res[torch.float32][k], res[torch.float64][k], name="%s_%s_vs_oracle" % (name, what))
            e_per = rel_err(per_object_i[k], res[torch.float64][k])
            assert ok[0] or (what == "g_pose" and ok[1] <= TRUTH_SLACK * e_per), (name, what, ok, e_per)


# S = 48 does not divide 256: a ray's rows can span a live and a dead super tile
@pytest.mark.parametrize("prec,S_", [("bf16", 64), ("bf16", 48), ("fp32", 64), ("fp32", 48)])
def test_dead_super_tiles_after_a_fully_live_backward(prec, S_):
    """Two backwards into ONE scratch buffer the test owns: every tile live first (every row's d xyz / d viewdir written), then a
    band of occ == 0 that kills whole super tiles.  The second backward's gradients equal the per-object render's and the oracle's."""
    im = 32
    S, sd, m, R, objs, lat, jit = _setup(prec, 3, im, S_, 410)
    live = [_all_live(o["mask_occ"]) for o in objs]
    first = _AbiBatch(S, m, R, objs, lat, jit, live, im, prec)
    scratch = torch.empty(first.scratch_bytes, dtype=torch.uint8, device=DEV)
    first.backward(scratch)
    band = [_band(o["mask_occ"], 6 + 2 * i, 22 + 2 * i) for i, o in enumerate(objs)]
    got = _AbiBatch(S, m, R, objs, lat, jit, band, im, prec).backward(scratch)
    assert all(bool(torch.isfinite(g).all()) for g in got)
    _check_vs_per_object("band_%s_S%d" % (prec, S_), S, m, R, objs, lat, jit, band, im, got)
    _check_vs_oracle("band_%s_S%d_obj0" % (prec, S_), prec, sd, objs[0], lat[0], jit[0], band[0], im, S_, [g[0] for g in got],
                     _per_object(S, m, R, objs[0], lat[0], jit[0], band[0], im))


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_object_without_live_rows_gets_zero_gradients(prec):
    """One object's occ is all zero: its gradients are exactly zero, the other objects' are unaffected."""
    im, S_ = 24, 64
    S, sd, m, R, objs, lat, jit = _setup(prec, 3, im, S_, 430)
    masks = [_all_live(o["mask_occ"]) for o in objs]
    masks[1] = torch.zeros_like(masks[1])
    got = _batched(S, m, R, objs, lat, jit, masks, im)
    for g in got:
        assert float(g[1].abs().max()) == 0.0
    for i in (0, 2):
        ref = _per_object(S, m, R, objs[i], lat[i], jit[i], masks[i], im)
        parity("%s_obj%d_g_shape" % (prec, i), got[1][i], ref[1], 1e-4)
        parity("%s_obj%d_g_texture" % (prec, i), got[2][i], ref[2], 1e-4)
        parity("%s_obj%d_g_pose" % (prec, i), got[0][i], ref[0], 1e-3)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_batch_without_live_rows(prec):
    """Every object's occ is zero: the decoder backward runs on an empty list and every gradient is exactly zero."""
    im, S_ = 16, 32
    S, sd, m, R, objs, lat, jit = _setup(prec, 2, im, S_, 450)
    _batched(S, m, R, objs, lat, jit, [_all_live(o["mask_occ"]) for o in objs], im)     # leave live-tile gradients in the scratch
    got = _batched(S, m, R, objs, lat, jit, [torch.zeros_like(o["mask_occ"]) for o in objs], im)
    for g in got:
        assert bool(torch.isfinite(g).all()) and float(g.abs().max()) == 0.0


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_poisoned_scratch_never_reaches_the_pose_gradient(prec):
    """snb_render_batch_bwd with a scratch buffer full of NaN and dead super tiles: the rays backward must not read the rows the
    decoder skipped.  The gradients are finite and equal the per-object render's (and the oracle's)."""
    im, S_ = 32, 48
    S, sd, m, R, objs, lat, jit = _setup(prec, 2, im, S_, 470)
    masks = [_band(o["mask_occ"], 4, 20 + 4 * i) for i, o in enumerate(objs)]
    ab = _AbiBatch(S, m, R, objs, lat, jit, masks, im, prec)
    got = ab.backward(torch.full((ab.scratch_bytes,), 255, dtype=torch.uint8, device=DEV))   # every float of the scratch NaN
    assert all(bool(torch.isfinite(g).all()) for g in got)
    _check_vs_per_object("poison_%s" % prec, S, m, R, objs, lat, jit, masks, im, got)
    _check_vs_oracle("poison_%s_obj0" % prec, prec, sd, objs[0], lat[0], jit[0], masks[0], im, S_, [g[0] for g in got],
                     _per_object(S, m, R, objs[0], lat[0], jit[0], masks[0], im))


def test_graphed_step_follows_the_occupancy_between_replays():
    """renderer.GraphedBatchStep replays one captured graph: the live list is rebuilt on the device every replay.  All tiles live
    on the first replay, a band of occ == 0 on the second (the pinned mask's content changes): each equals the call-by-call step."""
    im, S_ = 16, 32
    S, sd, m, R, objs, lat, jit = _setup("bf16", 3, im, S_, 490)
    pin = lambda t: t.contiguous().float().pin_memory()   # noqa: E731
    h_img = pin(torch.stack([o["img"] for o in objs]))
    h_mask = pin(torch.stack([_all_live(o["mask_occ"]) for o in objs]))
    h_cam, h_K = pin(torch.stack([o["cam_pose"] for o in objs])), pin(torch.stack([o["K"] for o in objs]))
    h_shp, h_tex = pin(torch.cat([l[0] for l in lat])), pin(torch.cat([l[1] for l in lat]))
    wlhs, rois = [o["wlh"] for o in objs], [o["roi"] for o in objs]
    jd = jit.to(DEV)
    step = S.renderer.GraphedBatchStep(R, m, DEV, h_img, h_mask, h_cam, wlhs, h_K, rois, h_shp, h_tex, im_sz=im, jitter=jd)
    for rep in range(2):
        if rep == 1:
            h_mask.copy_(torch.stack([_band(o["mask_occ"], 3, 12) for o in objs]))
        got = step.run()
        torch.cuda.synchronize()
        cam, shp, tex = [t.to(DEV).requires_grad_() for t in (h_cam, h_shp, h_tex)]
        rgb, dep, acc, tgt, occ = R.render_rays_batch(m, DEV, h_img, h_mask, cam, wlhs, h_K, rois, shp, tex, im_sz=im, jitter=jd)
        loss, parts = S.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)
        loss.backward(gradient=torch.ones(len(objs), device=DEV))
        ref = torch.cat([parts[:, :1], cam.grad.reshape(len(objs), 12), shp.grad, tex.grad], 1).cpu()
        parity("graph_rep%d_loss" % rep, got[:, 0], ref[:, 0], 1e-6)
        parity("graph_rep%d_g_pose" % rep, got[:, 1:13], ref[:, 1:13], 1e-4)
        parity("graph_rep%d_g_codes" % rep, got[:, 13:], ref[:, 13:], 1e-5)
