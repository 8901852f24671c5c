"""refine.SlotRefiner / refine.refine_stream: a stream of objects refined through fixed slots from one captured CUDA graph, and the
kernel generalisations under it (a step counter per slot with a guarded jitter-table read; AdamW on independent rows with their own
step counts, an active byte and the loss history)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import ADAM_OUTLIERS, parity_ok, rel_err
from oracle import oracle

DEV = "cuda"
BUDGETS = [6, 3, 6, 1, 4, 6, 2]      # 7 objects through 3 slots: slots are reused in the middle of the run
N_LIDAR = [37, 0, 64, 5, 64, 0, 12]   # 0 and the slot capacity (64) included
MAX_ITERS = 6


def snb():
    import supnerf_b200
    return supnerf_b200


def _model(prec):
    S = snb()
    m = S.SUPNeRF(3, 1, 3, 3, 256)
    m.load_state_dict({k: v.detach().clone() for k, v in oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=53).items()})
    m = m.to(DEV)
    m.precision = prec
    m.requires_grad_(False)
    return m


def _object(m, k, n_lidar=None, **kw):
    """ObjectRefiner k on its own seeds (object, latents, lidar pixels, jitter draws), as the BatchRefiner test builds them."""
    S = snb()
    import tools.refine_bench as rb
    seed = 80 + k
    obj = oracle.synthetic_object(seed, im_sz=32)
    shp0, tex0 = oracle.synthetic_latents(seed, 1)
    c2o = obj["cam_pose"]
    R_obj = c2o[:, :3].t().contiguous()
    t_obj = -(R_obj @ c2o[:, 3:]).reshape(3)
    rng = np.random.RandomState(seed)
    roi = [int(v) for v in obj["roi"]]
    n = N_LIDAR[k % len(N_LIDAR)] if n_lidar is None else n_lidar
    xy = (rng.randint(0, roi[2] - roi[0], n), rng.randint(0, roi[3] - roi[1], n)) if n else None
    torch.manual_seed(seed)
    args = dict(n_samples=64, im_sz=32, max_iters=MAX_ITERS, lidar_xy=xy)
    args.update(kw)
    return S.refine.ObjectRefiner(m, DEV, obj["img"], obj["mask_occ"], obj["K"], obj["roi"], np.linalg.norm(obj["wlh"]).astype(np.float32),
                                  shp0, tex0, rb.matrix_to_axis_angle(R_obj), t_obj, **args)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_stream_equals_per_object_refiners(prec):
    """refine_stream (7 objects, budgets 6 3 6 1 4 6 2, through 3 slots) against every object's own ObjectRefiner loop: each iteration's
    losses and loss_rgb2 (from loss_history), the lidar-pixel depths, and the optimised codes / pose parameters."""
    S = snb()
    m = _model(prec)
    seq = [_object(m, k) for k in range(len(BUDGETS))]
    hist = []
    for r, n in zip(seq, BUDGETS):
        h = []
        for _ in range(n):
            r.run(1)
            h.append(torch.cat([r.loss, r.loss_rgb2.reshape(1)]).clone())
        hist.append(torch.stack(h))
    objs = [_object(m, k) for k in range(len(BUDGETS))]
    out = S.refine.refine_stream(objs, BUDGETS, slots=3)
    assert [id(o) for o in out] == [id(o) for o in objs]
    tol1 = 1e-5 if prec == "fp32" else 1e-4
    tol = 1e-3 if prec == "fp32" else 5e-3
    for k, (r, ref) in enumerate(zip(out, seq)):
        assert tuple(r.loss_history.shape) == (BUDGETS[k], 4)
        assert torch.equal(r.loss_history[-1, :3], r.loss) and torch.equal(r.loss_history[-1, 3], r.loss_rgb2)
        for it in range(BUDGETS[k]):
            t = tol1 if it == 0 else tol
            assert parity_ok("obj%d_it%d_loss" % (k, it), r.loss_history[it, :3], hist[k][it, :3], t)
            assert parity_ok("obj%d_it%d_loss_rgb2" % (k, it), r.loss_history[it, 3], hist[k][it, 3], t)
        if N_LIDAR[k]:
            assert r.depth_pred.shape == ref.depth_pred.shape == (N_LIDAR[k],)
            assert parity_ok("obj%d_lidar_depth" % k, r.depth_pred, ref.depth_pred, tol1 if BUDGETS[k] == 1 else tol)
        assert parity_ok("obj%d_shapecode" % k, r.shapecode, ref.shapecode, 2e-2, outliers=ADAM_OUTLIERS)
        assert parity_ok("obj%d_texturecode" % k, r.texturecode, ref.texturecode, 2e-2, outliers=ADAM_OUTLIERS)
        assert parity_ok("obj%d_rot_vec" % k, r.rot_vec, ref.rot_vec, 5e-3) and parity_ok("obj%d_trans_vec" % k, r.trans_vec, ref.trans_vec, 5e-3)


def _slot_refiner(m, slots, **kw):
    return snb().refine.SlotRefiner(m, DEV, slots=slots, n_samples=64, im_sz=32, max_iters=MAX_ITERS, max_lidar=64, **kw)


@pytest.mark.gpu
def test_slot_graph_replay_equals_eager_steps():
    """The same stream through a captured SlotRefiner and through one that steps eagerly."""
    m = _model("bf16")
    eager = _slot_refiner(m, 3).stream([_object(m, k) for k in range(len(BUDGETS))], BUDGETS)
    graph = _slot_refiner(m, 3).capture().stream([_object(m, k) for k in range(len(BUDGETS))], BUDGETS)
    for k, (g, e) in enumerate(zip(graph, eager)):
        assert parity_ok("graph_loss_history_%d" % k, g.loss_history, e.loss_history, 1e-4)
        assert parity_ok("graph_shapecode_%d" % k, g.shapecode, e.shapecode, 2e-2, outliers=ADAM_OUTLIERS)


@pytest.mark.gpu
def test_admit_run_retire_without_host_synchronisation():
    m = _model("bf16")
    objs = [_object(m, k) for k in range(5)]
    sr = _slot_refiner(m, 2).capture()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        todo = list(zip(objs, [3, 1, 2, 2, 1]))[::-1]
        while todo or sr.busy():
            for _ in sr.free_slots():
                if todo:
                    sr.admit(*todo.pop())
            sr.run(1)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    sr.synchronize()
    assert sr.replays == 5 and abs(sr.idle_share() - 1 / 10) < 1e-12
    assert all(torch.isfinite(o.loss_history).all() for o in objs)


@pytest.mark.gpu
def test_adamw_rows_match_one_row_optimiser_and_torch():
    """Rows with different step counts and one inactive row: each active row is bit-identical to a one-row SlotAdamW on that row alone and
    within 1e-6 of torch.optim.AdamW on the CPU; the inactive row and its counter are bit-unchanged; the loss history row is written."""
    R = snb().refine
    g = torch.Generator().manual_seed(5)
    rows, sizes, lrs = 4, (256, 3), (0.02, 0.01)
    steps, active = [0.0, 3.0, 7.0, 1.0], [1, 1, 0, 1]
    P = [torch.randn(rows, n, generator=g) for n in sizes]
    G = [torch.randn(rows, n, generator=g) * 1e-2 for n in sizes]
    M = [torch.randn(rows, n, generator=g) * 1e-2 for n in sizes]
    V = [torch.rand(rows, n, generator=g) * 1e-4 for n in sizes]
    params = [p.to(DEV) for p in P]
    opt = R.SlotAdamW([{"params": p, "lr": lr} for p, lr in zip(params, lrs)], rows=rows)
    for i in range(2):
        params[i].grad = G[i].to(DEV)
        opt.m[i].copy_(M[i])
        opt.v[i].copy_(V[i])
    opt.step_t.copy_(torch.tensor(steps))
    opt.active.copy_(torch.tensor(active, dtype=torch.uint8))
    loss3 = torch.randn(rows, 3, generator=g).to(DEV)
    eval3 = torch.randn(rows, 3, generator=g).to(DEV)
    history = torch.full((rows, 8, 4), -1.0, device=DEV)
    opt.step(loss3, eval3[:, 1], history)
    torch.cuda.synchronize()
    for r in range(rows):
        if not active[r]:
            assert all(torch.equal(params[i][r].cpu(), P[i][r]) and torch.equal(opt.m[i][r].cpu(), M[i][r]) and
                       torch.equal(opt.v[i][r].cpu(), V[i][r]) for i in range(2))
            assert opt.step_t[r].item() == steps[r] and bool((history[r] == -1).all())
            continue
        one = [P[i][r].clone().to(DEV) for i in range(2)]
        ref = R.SlotAdamW([{"params": p, "lr": lr} for p, lr in zip(one, lrs)], rows=1)
        for i in range(2):
            one[i].grad = G[i][r].to(DEV)
            ref.m[i].copy_(M[i][r])
            ref.v[i].copy_(V[i][r])
        ref.step_t.fill_(steps[r])
        ref.step()
        cpu = [P[i][r].clone().requires_grad_() for i in range(2)]
        topt = torch.optim.AdamW([{"params": [p], "lr": lr} for p, lr in zip(cpu, lrs)])
        for i in range(2):
            cpu[i].grad = G[i][r].clone()
            topt.state[cpu[i]] = {"step": torch.tensor(steps[r]), "exp_avg": M[i][r].clone(), "exp_avg_sq": V[i][r].clone()}
        topt.step()
        for i in range(2):
            assert torch.equal(params[i][r], one[i]) and torch.equal(opt.m[i][r], ref.m[i]) and torch.equal(opt.v[i][r], ref.v[i])
            assert rel_err(params[i][r], cpu[i]) <= 1e-6
        assert opt.step_t[r].item() == steps[r] + 1 == ref.step_t.item()
        s = int(steps[r])
        assert torch.equal(history[r, s, :3], loss3[r]) and history[r, s, 3].item() == eval3[r, 1].item()
        assert bool((history[r, :s] == -1).all()) and bool((history[r, s + 1:] == -1).all())


def _pose_fwd(rot, trans, jitter, jitter2, T, steps, active, err, obj_diag):
    """snb_refine_pose_slots_fwd with steps (C,)."""
    from supnerf_b200 import _lib
    from supnerf_b200._lib import ptr, stream_ptr
    lib = _lib.load()
    c, s = rot.shape[0], jitter.shape[-1]
    cam = torch.empty(c, 3, 4, device=DEV)
    z, z2 = torch.empty(c, s, device=DEV), torch.empty(c, s, device=DEV)
    rc = lib.snb_refine_pose_slots_fwd(ptr(rot), ptr(trans), c, 0, ptr(obj_diag), s, ptr(jitter), ptr(jitter2), ptr(steps), T, ptr(active),
                                       ptr(err), ptr(cam), ptr(z), ptr(z2), stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()
    return cam, z, z2


@pytest.mark.gpu
def test_slot_counter_guard():
    """The jitter tables hold T + 1 rows per slot but are passed as T rows, so an unguarded read at row T would read valid memory: an
    active slot at counter T (or -1) gets NaN z / z2 and sets the flag; inactive, the same slot gives finite z and no flag."""
    snb()
    g = torch.Generator().manual_seed(9)
    c, T, s = 4, 5, 64
    rot = (torch.randn(c, 3, generator=g) * 0.3).to(DEV)
    trans = (torch.randn(c, 3, generator=g) + torch.tensor([0.0, 0.0, 6.0])).to(DEV)
    jit = torch.rand(c, T + 1, s, generator=g).to(DEV)
    jit2 = torch.rand(c, T + 1, s, generator=g).to(DEV)
    obj_diag = torch.full((c,), 2.0, device=DEV)
    steps = torch.tensor([0.0, float(T), 2.0, -1.0], device=DEV)
    err = torch.zeros(1, dtype=torch.int32, device=DEV)
    _, z, z2 = _pose_fwd(rot, trans, jit, jit2, T, steps, torch.ones(c, dtype=torch.uint8, device=DEV), err, obj_diag)
    assert int(err.item()) == 1
    for b, bad in enumerate([False, True, False, True]):
        assert bool(torch.isnan(z[b]).all()) == bad and bool(torch.isnan(z2[b]).all()) == bad
        assert bad or bool(torch.isfinite(z[b]).all() and torch.isfinite(z2[b]).all())
    err.zero_()
    _, z, z2 = _pose_fwd(rot, trans, jit, jit2, T, steps, torch.tensor([1, 0, 1, 0], dtype=torch.uint8, device=DEV), err, obj_diag)
    assert int(err.item()) == 0 and bool(torch.isfinite(z).all() and torch.isfinite(z2).all())


@pytest.mark.gpu
def test_admit_rejects_what_the_slots_cannot_hold():
    m = _model("bf16")
    sr = snb().refine.SlotRefiner(m, DEV, slots=1, n_samples=64, im_sz=32, max_iters=4, max_lidar=8)
    with pytest.raises(ValueError):
        sr.admit(_object(m, 1, lr_shape=0.05), 2)                # other optimiser settings
    with pytest.raises(ValueError):
        sr.admit(_object(m, 1, n_samples=32), 2)                 # other sample count
    with pytest.raises(ValueError):
        sr.admit(_object(m, 1), 5)                               # budget > max_iters
    with pytest.raises(ValueError):
        sr.admit(_object(m, 1, max_iters=2), 3)                  # budget > the object's jitter rows
    with pytest.raises(ValueError):
        sr.admit(_object(m, 0, n_lidar=9), 2)                    # more lidar pixels than the slot capacity
    assert sr.admit(_object(m, 0, n_lidar=8), 2) == 0
    with pytest.raises(ValueError):
        sr.admit(_object(m, 1), 2)                               # no free slot


def test_slot_refiner_has_no_cpu_path():
    S = snb()
    with pytest.raises(RuntimeError):
        S.refine.SlotRefiner(S.SUPNeRF(3, 1, 3, 3, 256), "cpu")
