#!/usr/bin/env python
"""Refining an evaluation split: N objects x `iters` refine iterations (optimize_objs_w_pose_unified, optimizer_nuscenes.py:684-769), in two
modes alternated in one process, each timed from the first ObjectRefiner construction to the final synchronisation:
  groups : ObjectRefiners -> refine.BatchRefiner of C -> capture() -> run(iters) -> write_back(), group after group (every group pays the
           warm-up, the capture and its device synchronisation);
  stream : refine.SlotRefiner of C slots, captured once, objects admitted and retired between replays (what refine.refine_stream runs).
Per mode: wall time, objects/s, ms per object-iteration, device time from CUDA events (whole window, and the refine iterations alone), the
share of slot-iterations that ran idle, and the per-object losses of both modes compared.  The card name and power limit are read (query
only) in the same call and printed beside the numbers.
  python tools/refine_stream_bench.py [--objects 256] [--iters 50] [--slots 16] [--runs 3] [--precisions bf16,fp32]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import supnerf_b200 as snb  # noqa: E402
from supnerf_b200 import synthetic  # noqa: E402
from tools.refine_bench import matrix_to_axis_angle  # noqa: E402


def card(dev):
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        if r.returncode == 0 and r.stdout.strip():
            name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
            info.update(name=name, power_limit=power, max_sm_clock=clock)
    except (OSError, subprocess.SubprocessError, ValueError):
        info["power_limit"] = "not readable"
    return info


def inputs(n, im, dev):
    """The objects' inputs (what the reference's DataLoader delivers): built once, outside the timed windows."""
    objs = []
    for i in range(n):
        o = synthetic.synthetic_object(300 + i, im_sz=im)
        s, t = synthetic.synthetic_latents(300 + i, 1)
        c2o = o["cam_pose"]
        R_obj = c2o[:, :3].t().contiguous()
        objs.append(dict(img=o["img"].to(dev), mask=o["mask_occ"].to(dev), K=o["K"].to(dev), roi=o["roi"],
                         obj_diag=np.linalg.norm(o["wlh"]).astype(np.float32), shapecode=s.to(dev), texturecode=t.to(dev),
                         rot_vec=matrix_to_axis_angle(R_obj).to(dev), trans_vec=(-(R_obj @ c2o[:, 3:])).reshape(3).to(dev)))
    return objs


def refiners(model, dev, objs, a, iters):
    out = []
    for i, o in enumerate(objs):
        torch.manual_seed(1000 + i)
        out.append(snb.refine.ObjectRefiner(model, dev, o["img"], o["mask"], o["K"], o["roi"], o["obj_diag"], o["shapecode"], o["texturecode"],
                                            o["rot_vec"], o["trans_vec"], n_samples=a.samples, im_sz=a.im, max_iters=iters))
    return out


def run_mode(mode, model, dev, objs, a, iters):
    n, c = len(objs), a.slots
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    refs = refiners(model, dev, objs, a, iters)
    t_built = time.perf_counter()
    windows, idle = [], 0.0
    if mode == "groups":
        for g in range(0, n, c):
            bat = snb.refine.BatchRefiner(refs[g:g + c]).capture()
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record()
            bat.run(iters)
            w1.record()
            bat.write_back()
            windows.append((w0, w1))
    else:
        sr = snb.refine.SlotRefiner(model, dev, slots=c, n_samples=a.samples, im_sz=a.im, max_iters=iters).capture()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        sr.stream(refs, iters)                  # ends with a synchronisation
        w1.record()
        windows.append((w0, w1))
        idle = sr.idle_share()
    ev1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    iters_ms = sum(x.elapsed_time(y) for x, y in windows)
    res = {"wall_ms": wall, "objects_per_s": n / (wall / 1e3), "ms_per_object_iteration": wall / (n * iters),
           "device_ms_events": ev0.elapsed_time(ev1), "refine_iterations_ms_events": iters_ms,
           "refine_iterations_ms_per_object_iteration": iters_ms / (n * iters), "construct_ms": (t_built - t0) * 1e3, "idle_share": idle}
    if mode == "groups":
        res["groups"] = len(windows)
        res["setup_ms_per_group"] = (wall - res["construct_ms"] - iters_ms) / len(windows)
    losses = torch.stack([r.loss.detach().reshape(3) for r in refs]).cpu()
    return res, losses


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--objects", type=int, default=256)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--slots", type=int, default=16)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--im", type=int, default=32)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--precisions", default="bf16,fp32")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("refine_stream_bench needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    objs = inputs(a.objects, a.im, dev)
    result = {"workload": "%d objects x %d refine iterations, %dx%d rays x %d samples, SUPNeRF(3,1,3,3,256), %d slots / objects per group"
                          % (a.objects, a.iters, a.im, a.im, a.samples, a.slots), "card": card(dev), "runs": a.runs, "precisions": {}}
    for prec in a.precisions.split(","):
        model = snb.SUPNeRF(3, 1, 3, 3, 256)
        model.load_state_dict(synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=3))
        model = model.to(dev)
        model.precision = prec
        model.requires_grad_(False)
        for mode in ("groups", "stream"):     # warm-up: module loads, weight packing, allocator
            run_mode(mode, model, dev, objs[:a.slots], a, 3)
        runs, losses = {"groups": [], "stream": []}, {}
        for _ in range(a.runs):
            for mode in ("groups", "stream"):
                r, l_ = run_mode(mode, model, dev, objs, a, a.iters)
                runs[mode].append(r)
                losses.setdefault(mode, l_)
        tol = 5e-3 if prec == "bf16" else 1e-3
        err = rel(losses["stream"], losses["groups"])
        summary = {}
        for mode, rs in runs.items():
            summary[mode] = {k: round(statistics.median(r[k] for r in rs), 4) for k in rs[0]}
            summary[mode]["wall_ms_all_runs"] = [round(r["wall_ms"], 2) for r in rs]
        summary["stream_speedup_wall"] = round(summary["groups"]["wall_ms"] / summary["stream"]["wall_ms"], 3)
        summary["losses_stream_vs_groups"] = {"max_rel_err": err, "tol": tol, "match": err <= tol}
        result["precisions"][prec] = summary
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
