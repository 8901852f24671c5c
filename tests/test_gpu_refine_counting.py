"""The refiners' host-side iteration count and their warm-up before capture: run() refuses, before it issues anything, an iteration
past the pre-drawn jitter tables (also after direct step() calls), capture() works with tables shorter than the warm-up, and the
batched capture leaves the refine state bit for bit as it found it."""
import numpy as np
import pytest
import torch

from conftest import ADAM_OUTLIERS, parity_ok
from oracle import oracle

pytestmark = pytest.mark.gpu
DEV = "cuda"
N_LIDAR = [37, 0, 64, None]   # 0: an empty lidar list; None: no lidar evaluation


def snb():
    import supnerf_b200
    return supnerf_b200


def _model():
    m = snb().SUPNeRF(3, 1, 3, 3, 256)
    m.load_state_dict({k: v.detach().clone() for k, v in oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=53).items()})
    m = m.to(DEV)
    m.precision = "fp32"
    m.requires_grad_(False)
    return m


def _object(m, k, max_iters, fused=True):
    """ObjectRefiner k on its own seeds (object, latents, lidar pixels, jitter draws): two calls give identical twins."""
    import tools.refine_bench as rb
    seed = 110 + k
    obj = oracle.synthetic_object(seed, im_sz=32)
    shp0, tex0 = oracle.synthetic_latents(seed, 1)
    c2o = obj["cam_pose"]
    R_obj = c2o[:, :3].t().contiguous()
    t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
    rng = np.random.RandomState(seed)
    roi = [int(v) for v in obj["roi"]]
    n = N_LIDAR[k % len(N_LIDAR)]
    xy = None if n is None else (rng.randint(0, roi[2] - roi[0], n), rng.randint(0, roi[3] - roi[1], n))
    torch.manual_seed(seed)
    return snb().refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                      shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, n_samples=64, im_sz=32, max_iters=max_iters,
                                      fused=fused, lidar_xy=xy)


def _state(r):
    """Every tensor an issued iteration would change: parameters and the optimiser's moments and step counters."""
    ts = [r.shapecode, r.texturecode, r.rot_vec, r.trans_vec]
    return [t.detach().clone() for t in ts + r.opt.m + r.opt.v + [r.opt.step_t]]


def _launches():
    return snb()._lib.load().snb_launch_count()


@pytest.mark.parametrize("kind", ["object", "batch"])
@pytest.mark.parametrize("graphed", [False, True])
def test_run_past_the_jitter_table_raises_and_issues_nothing(kind, graphed):
    """run(k) then run(max_iters - k + 1), and step() then a run() that would cross the table: ValueError with no launch, no state
    change and no count taken; what is left of the table still runs."""
    m = _model()
    T, k = 5, 2
    make = (lambda: _object(m, 0, T)) if kind == "object" else (lambda: snb().refine.BatchRefiner([_object(m, j, T) for j in range(3)]))
    for first in ("run", "step"):
        r = make()
        if graphed:
            r.capture()
        for _ in range(k):
            r.run(1) if first == "run" else r.step()
        torch.cuda.synchronize()
        before, n0 = _state(r), _launches()
        with pytest.raises(ValueError):
            r.run(T - k + 1)
        assert _launches() == n0 and all(torch.equal(a, b) for a, b in zip(_state(r), before))
        r.run(T - k)
        with pytest.raises(ValueError):
            r.step()
        torch.cuda.synchronize()
        assert bool(torch.isfinite(r.loss).all())
        assert torch.equal(r.opt.step_t.cpu(), torch.full_like(r.opt.step_t.cpu(), float(T)))


def _one_iteration_close(name, a, b):
    """A captured first iteration against a fresh twin's eager one: losses to 1e-5 (fp32), the updated parameters to the trajectory
    tolerances of AdamW's first step (~ lr * sign(g))."""
    assert parity_ok(name + "_loss", a.loss, b.loss, 1e-5) and parity_ok(name + "_loss_rgb2", a.loss_rgb2, b.loss_rgb2, 1e-5)
    assert parity_ok(name + "_shapecode", a.shapecode, b.shapecode, 2e-2, outliers=ADAM_OUTLIERS)
    assert parity_ok(name + "_rot_vec", a.rot_vec, b.rot_vec, 5e-3) and parity_ok(name + "_trans_vec", a.trans_vec, b.trans_vec, 5e-3)


@pytest.mark.parametrize("fused", [True, False])
def test_object_refiner_capture_with_fewer_jitter_rows_than_warmup_steps(fused):
    m = _model()
    cap = _object(m, 0, 1, fused=fused).capture()          # warmup=3 > max_iters=1
    cap.run(1)
    twin = _object(m, 0, 1, fused=fused)
    twin.step()
    torch.cuda.synchronize()
    _one_iteration_close("object", cap, twin)
    assert cap.depth_pred.shape == twin.depth_pred.shape and parity_ok("object_lidar_depth", cap.depth_pred, twin.depth_pred, 1e-5)
    with pytest.raises(ValueError):
        cap.run(1)


def test_object_group_capture_with_fewer_jitter_rows_than_warmup_steps():
    m = _model()
    grp = snb().refine.ObjectGroup([_object(m, j, 1) for j in range(3)]).capture()
    grp.run(1)
    twins = [_object(m, j, 1) for j in range(3)]
    for t in twins:
        t.step()
    torch.cuda.synchronize()
    for j, (a, b) in enumerate(zip(grp.refiners, twins)):
        _one_iteration_close("group%d" % j, a, b)
    with pytest.raises(ValueError):
        grp.run(1)


def test_batch_refiner_capture_with_fewer_jitter_rows_than_warmup_steps():
    m = _model()
    cap = snb().refine.BatchRefiner([_object(m, j, 1) for j in range(4)]).capture()
    cap.run(1)
    twin = snb().refine.BatchRefiner([_object(m, j, 1) for j in range(4)])
    twin.step()
    cap.synchronize()           # raises if a slot read outside its jitter table
    assert parity_ok("batch_loss", cap.loss, twin.loss, 1e-5) and parity_ok("batch_loss_rgb2", cap.loss_rgb2, twin.loss_rgb2, 1e-5)
    assert parity_ok("batch_shapecode", cap.shapecode, twin.shapecode, 2e-2, outliers=ADAM_OUTLIERS)
    assert parity_ok("batch_rot_vec", cap.rot_vec, twin.rot_vec, 5e-3) and parity_ok("batch_trans_vec", cap.trans_vec, twin.trans_vec, 5e-3)
    for b, (d, e) in enumerate(zip(cap.lidar_depths(), twin.lidar_depths())):
        if N_LIDAR[b]:
            assert d.shape == e.shape == (N_LIDAR[b],) and parity_ok("batch_lidar_depth", d, e, 1e-5)
        else:
            assert d is None and e is None                  # empty lidar list and no lidar evaluation alike
    with pytest.raises(ValueError):
        cap.run(1)


def test_batch_refiner_capture_leaves_the_refine_state_bit_identical():
    """Captured after two eager iterations (non-zero moments and counters): parameters, moments, step counters, active bytes and loss
    history unchanged to the bit, and the error flag clear."""
    m = _model()
    bat = snb().refine.BatchRefiner([_object(m, j, 4) for j in range(4)])
    bat.run(2)
    torch.cuda.synchronize()
    before = _state(bat) + [bat.opt.active.clone(), bat.history.clone()]
    bat.capture()
    bat.synchronize()
    after = _state(bat) + [bat.opt.active, bat.history]
    assert all(torch.equal(a, b) for a, b in zip(after, before))
    assert bat.lidar_depths()[1] is None and bat.lidar_depths()[3] is None
