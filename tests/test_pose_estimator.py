"""SURVEY 8f rank 2, the pose-estimator forward: supnerf_b200.pose_estimator / SUPNeRF.encode_img / pose_update against outputs of the
UNMODIFIED reference (tests/golden/pose_estimator.npz, tools/make_golden.py:golden_pose_estimator).  The encoder is plain torch
(cuDNN / CPU convolutions): its tests run on the CPU too; the joint training step needs the decoder kernels (-m gpu).
The image and weight gradients of the fixture are stored as a strided sample of 1/2 .. 1/17 of their elements (conftest.Sampled):
they are judged on those elements, against max|.| of the whole array."""
import numpy as np
import pytest
import torch

from conftest import T, load_golden, parity, rel_err

TOL = 1e-5


def _model(g, device="cpu"):
    import supnerf_b200 as snb
    from supnerf_b200 import synthetic
    m = snb.SUPNeRF(3, 1, 3, 3, 256)
    m.materialize_pose_estimator()
    sd = dict(synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=int(g["seed"])))
    sd.update(synthetic.pose_estimator_state(m.state_dict(), int(g["seed"])))
    res = m.load_state_dict(sd)
    assert not res.missing_keys and not res.unexpected_keys
    return m.to(device)


def test_state_dict_keys_of_the_materialised_module_match_the_reference():
    import json
    import os
    from conftest import ROOT
    import supnerf_b200 as snb
    keys = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_keys.json")))["SUPNeRF_3_1_3_3_256"]
    m = snb.SUPNeRF(3, 1, 3, 3, 256)
    assert not m.has_pose_estimator() and len(m.state_dict()) == 28          # decoder-only until the pose estimator is used
    m.materialize_pose_estimator()
    sd = m.state_dict()
    assert list(sd.keys()) == list(keys.keys())
    assert all(list(sd[k].shape) == keys[k][0] for k in keys)
    assert abs(sum(p.numel() for p in m.parameters()) - 49.03e6) < 0.05e6


def test_reference_checkpoint_entries_move_into_the_materialised_modules():
    """A reference checkpoint loaded BEFORE the pose estimator exists keeps its encoder entries (strict load, models.py) and hands
    them to the modules on first use."""
    import supnerf_b200 as snb
    g = load_golden("pose_estimator")
    full = _model(g).state_dict()
    m = snb.SUPNeRF(3, 1, 3, 3, 256)
    res = m.load_state_dict(full)
    assert not res.missing_keys and not res.unexpected_keys and not m.has_pose_estimator()
    m.eval()
    with torch.no_grad():
        out = m.encode_img(T(g["img"]))
    assert m.has_pose_estimator() and rel_err(out[2], g["eval_pose"]) < TOL
    assert set(m.state_dict().keys()) == set(full.keys())


def test_encode_img_and_pose_update_against_the_reference_cpu():
    g = load_golden("pose_estimator")
    m = _model(g)
    m.eval()
    img = T(g["img"]).requires_grad_()
    f_s, f_t, f_p, uv, wlh = m.encode_img(img)
    assert wlh is None
    delta = m.pose_update(f_p, T(g["uv_src"]))
    for name, t in (("shape", f_s), ("texture", f_t), ("pose", f_p), ("uv", uv), ("delta", delta)):
        assert rel_err(t, g["eval_" + name]) < TOL, name
    sum((t * T(g["up_" + n_])).sum() for t, n_ in zip((f_s, f_t, f_p, uv, delta), ("shape", "texture", "pose", "uv", "delta"))).backward()
    assert rel_err(img.grad, g["eval_g_img"]) < TOL
    enc = m.img_encoder
    for name, t in (("conv1", enc.conv1.weight.grad), ("fc_pose", enc.fc_pose.weight.grad), ("out_delta", m.out_delta_layer.weight.grad),
                    ("regress0", m.regress_layer_0[0].weight.grad), ("l4pose_conv", enc.layer4_pose[2].conv2.weight.grad[::16, ::16])):
        assert rel_err(t, g["eval_gw_" + name]) < TOL, name
    m.train()      # batch statistics + running-stat update
    with torch.no_grad():
        f_s, f_t, f_p, uv, _ = m.encode_img(T(g["img"]))
    for name, t in (("shape", f_s), ("texture", f_t), ("pose", f_p), ("uv", uv)):
        assert rel_err(t, g["train_" + name]) < TOL, name
    assert rel_err(enc.bn1.running_mean, g["train_running_mean_bn1"]) < TOL


def test_box_corner_projection_helpers_against_the_reference():
    from supnerf_b200 import pose_estimator as pe
    g = load_golden("pose_estimator")
    pose, wlh, K, roi = T(g["obj_pose"]), T(g["wlh"]), T(g["K"]), T(g["roi"])
    corners = pe.corners_of_box_batch(pose, wlh)
    assert rel_err(corners, g["corners"]) < 1e-6
    assert rel_err(pe.corners_of_box_batch(pose, wlh, is_kitti=True, scale=1.1), g["corners_kitti"]) < 1e-6
    uv = pe.view_points_batch(corners, K, normalize=True)
    assert rel_err(uv, g["uv_all"]) < 1e-6
    n1, dim = pe.normalize_by_roi(uv[:, :2, :], roi, need_square=True)
    n2, none = pe.normalize_by_roi(uv[:, :2, :], roi, need_square=False)
    assert rel_err(n1, g["uv_norm"]) < 1e-6 and rel_err(dim, g["uv_dim"]) == 0 and none is None and rel_err(n2, g["uv_norm_nonsquare"]) < 1e-6
    # the axis-angle maps (pytorch3d's in the reference; parity unpinned): inverse of one another, proper rotations
    v = torch.tensor([[0.3, -1.1, 0.7], [1e-4, 2e-4, -1e-4], [2.0, 0.1, -0.4]])
    R = pe.axis_angle_to_matrix_batch(v)
    assert rel_err(R @ R.transpose(1, 2), torch.eye(3).expand(3, 3, 3)) < 1e-6 and rel_err(pe.matrix_to_axis_angle_batch(R), v) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("prec,tol", [("fp32", 1e-5), ("bf16", 2e-2)])
def test_joint_training_step_against_the_reference_gpu(prec, tol):
    """ParallelModel.forward + backward (trainer_unified_nuscenes.py:27-148): encoder + pose regression x3 + the decoder /
    compositing kernels + every loss, gradients to codes, encoder and decoder weights.  `prec` selects the decoder back end.
    Pass 1 (judged): the image encoder runs on the CPU, i.e. bit-identically to the reference run that made the fixture, so the
    codes entering the decoder kernels are the reference's and their gradients are held to the stated tolerance (fp64 truth from
    the same reference run in float64 for the ill-conditioned sums).  Pass 2 (recorded): the whole step on the GPU with the cuDNN
    fp32 encoder (TF32 off) -- train-mode batch norm over 2 images makes the encoder's codes differ by ~1e-5 from the CPU's, which
    the code gradients amplify ~100x; losses and predictions are still held to 1e-4."""
    import copy
    from supnerf_b200 import pose_estimator as pe
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g = load_golden("pose_estimator")
    dev = "cuda:0"
    hp = {"loss_pose_coef": 0.01, "loss_code_coef": 0.1, "loss_occ_coef": 0.1}
    D = lambda k: T(g[k], device=dev)   # noqa: E731
    for enc_on_cpu in (True, False):
        m = _model(g, dev)
        m.precision = prec
        m.train()
        enc_cpu = copy.deepcopy(m.img_encoder).cpu() if enc_on_cpu else None
        shp, tex = D("j_shapecode").requires_grad_(), D("j_texturecode").requires_grad_()

        def encode(img, enc_cpu=enc_cpu):
            out = enc_cpu(img.cpu(), m.pose_shortcut)
            return tuple(t.to(dev) for t in out) + (None,)
        losses_all, total, shp_o, tex_o, pose3, uv_direct = pe.joint_training_losses(
            m, hp, D("img"), shp, tex, D("j_xyz"), D("j_viewdir"), D("j_z_vals"), D("j_rgb_tgt"), D("j_occ"), D("j_src_pose"), D("j_tgt_uv"),
            D("roi"), D("K"), D("wlh"), D("j_tgt_uv"), encode=encode if enc_on_cpu else None)
        total.mean().backward()
        tag = "" if enc_on_cpu else "cudnn_encoder_"
        for k in ("loss_pose_direct", "loss_code", "loss_pose_iter1", "loss_pose_iter2", "loss_pose_iter3", "loss_rgb", "loss_occ", "loss_reg", "loss_total"):
            parity(tag + k, losses_all[k], g["j_" + k], tol if k in ("loss_rgb", "loss_occ", "loss_total") else 1e-4)
        parity(tag + "pred_pose3", pose3, g["j_pred_pose3"], 1e-4)
        parity(tag + "pred_uv_direct", uv_direct, g["j_pred_uv_direct"], 1e-4)
        parity(tag + "shapecode_out", shp_o, g["j_shapecode_out"], 1e-4)
        enc = enc_cpu if enc_on_cpu else m.img_encoder
        grads = (("g_shapecode", shp.grad), ("g_texturecode", tex.grad), ("gw_conv1", enc.conv1.weight.grad), ("gw_fc_shape", enc.fc_shape.weight.grad),
                 ("gw_out_delta", m.out_delta_layer.weight.grad), ("gw_encoding_xyz", m.encoding_xyz[0].weight.grad), ("gw_rgb2", m.rgb[2].weight.grad))
        for name, t in grads:
            parity(tag + name, t, g["j_" + name], tol, truth=g["j64_" + name], info=not enc_on_cpu)
