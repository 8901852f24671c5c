#!/usr/bin/env python
"""Benchmark of the SUP-NeRF render hot path (BASELINE.json metric: rays/s fwd+bwd, CodeNeRF-MLP render).

Workload at N=1 = BASELINE.json configs[1]: AutoRF-mix (3/1/256) render fwd+bwd of a batch of 16 synthetic car
objects at 128x128 patches (16 384 rays/object, 64 samples/ray).  One STEP = all 16 objects: for each object the
reference's NeRFRenderer.render_rays pipeline (rays -> slab test -> stratified samples -> decoder -> compositing),
the refine losses and the backward pass to the camera pose and both latent codes (weights frozen: refine mode).
N>1: object-parallel, every rank renders its own 16 objects (weak scaling, no collective on the data path).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|fp32] [--dump-outputs DIR]

`value`   : rays/s with every input already resident in HBM (device tensors in, loss stays on device).
`e2e`     : the same through the public drop-in API NeRFRenderer.render_rays with HOST inputs (pinned img / mask /
            pose / latents copied H2D every step, loss + gradients read back D2H every step).
`--impl reference`: the reference's algorithm on the host cores (the CPU oracle port, all threads), same metric, on a
            bounded sample of the workload (one object, 64x64 rays per step).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_OBJ, IM_SZ, N_SAMPLES = 16, 128, 64
MAC_PER_SAMPLE = 449664  # BASELINE.md: decoder Bs=3, Bt=1, W=256
METRIC = "rays/s fwd+bwd, CodeNeRF-MLP render"
WORKLOAD = "configs[1]: AutoRF-mix (3/1/256) render fwd+bwd, 16 objects x 128x128 rays x 64 samples per GPU per step"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), tf_burst=d["bf16_tflops"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_sustained=1400.0, tf_burst=1590.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, 20 ms period; nvidia-smi fallback)."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index, self.sm, self.mx, self.reasons, self.n = index, [], None, set(), 0
        self.stop = threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def sample(self):
        if self.nvml is not None:
            self.sm.append(float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)))
            r = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(self.nvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                else int(self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            for name, bit in self.BAD.items():
                if r & bit:
                    self.reasons.add(name)
        else:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=5).stdout.strip()
            c = [x.strip() for x in out.split(",")]
            self.sm.append(float(c[0]))
            self.mx = float(c[1])
            for i, name in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
                if c[2 + i].lower().startswith("active"):
                    self.reasons.add(name)
        self.n += 1

    def run(self):
        while not self.stop.is_set():
            try:
                self.sample()
            except Exception:
                pass
            self.stop.wait(0.02 if self.nvml is not None else 0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=3)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_min_mhz": float(min(self.sm)) if self.sm else None,
                "sm_max_mhz": self.mx, "reasons": sorted(self.reasons), "samples": self.n,
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def make_objects(seed0, n_obj, im_sz):
    from supnerf_b200 import synthetic  # seeded input generators shared with the tests: CPU and GPU arms see the same bits
    objs = []
    for i in range(n_obj):
        o = synthetic.synthetic_object(seed0 + i, im_sz=im_sz)
        s, t = synthetic.synthetic_latents(seed0 + i, 1)
        o["shapecode"], o["texturecode"] = s, t
        objs.append(o)
    return objs


# what one step of the timed path hands its caller, per object, with the shape each is written in by --dump-outputs
OUTPUTS = {"rgb": (N_OBJ, -1, 3), "depth": (N_OBJ, -1), "acc": (N_OBJ, -1), "loss": (N_OBJ,), "cam_pose_grad": (N_OBJ, 3, 4),
           "shapecode_grad": (N_OBJ, -1), "texturecode_grad": (N_OBJ, -1)}


def dump_outputs(path, last):
    """DIR/<name>.npy (float32) for every output of the last timed step: 16 objects x 128 x 128 rays, 5.3 MB in all."""
    os.makedirs(path, exist_ok=True)
    for name, shape in OUTPUTS.items():
        t = last[name]
        t = torch.stack(t) if isinstance(t, list) else t
        np.save(os.path.join(path, name + ".npy"), t.detach().reshape(shape).float().cpu().numpy())


def refine_loss(rgb, acc, tgt, occ):
    """optimizer_nuscenes.py:729-736"""
    den = torch.sum(torch.abs(occ)) + 1e-9
    loss_rgb = torch.sum((rgb - tgt) ** 2 * torch.abs(occ)) / den
    loss_occ = torch.sum(torch.exp(-occ * (0.5 - acc.unsqueeze(-1))) * torch.abs(occ)) / den
    return loss_rgb + 0.1 * loss_occ


# ----------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import supnerf_b200 as snb
    from supnerf_b200 import _lib, ops, synthetic

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line (NCCL_DEBUG=VERSION prints a banner)
        import datetime
        # a short collective timeout: a mismatched collective must fail in minutes, not hold the GPUs for the default 10
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=150))
    lib = _lib.load()

    sd = synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=0)
    model = snb.AutoRFMix(shape_blocks=3, texture_blocks=1, latent_dim=256)
    model.load_state_dict(sd)
    model = model.to(dev)
    model.precision = args.precision
    model.requires_grad_(False)  # refine mode: weights frozen (stated in config)
    R = snb.renderer.NeRFRenderer(n_samples=N_SAMPLES)
    # weak scaling with IDENTICAL per-GPU work: every rank renders its own copy of the same 16-object set (the objects' hit
    # fractions differ by 2.5x, so rank-dependent sets would measure load imbalance rather than the system)
    objs = make_objects(100, N_OBJ, IM_SZ)
    n_rays = IM_SZ * IM_SZ

    # device-resident copies (for `value`) and pinned host copies (for `e2e`)
    dobjs, hobjs = [], []
    for o in objs:
        # crop already at im_sz: the reference's Resize is the identity here
        dobjs.append(dict(K=o["K"].to(dev), cam=o["cam_pose"].to(dev).requires_grad_(), wlh=o["wlh"], roi=o["roi"],
                          img=o["img"].to(dev), mask=o["mask_occ"].to(dev),
                          shp=o["shapecode"].to(dev).requires_grad_(), tex=o["texturecode"].to(dev).requires_grad_()))
        hobjs.append(dict(K=o["K"].pin_memory(), cam=o["cam_pose"].pin_memory(), wlh=o["wlh"], roi=o["roi"], img=o["img"].pin_memory(),
                          mask=o["mask_occ"].pin_memory(), shp=o["shapecode"].pin_memory(), tex=o["texturecode"].pin_memory()))
    fp32_tc = args.precision == "fp32" and snb.ops.FP32_TENSOR_CORES      # fp32 mode on the split-precision tensor-core kernels
    batched = args.batched and (args.precision == "bf16" or fp32_tc)

    # Objects are independent (SURVEY 8e).  Default: ALL 16 objects of the step go through ONE launch set (NeRFRenderer.render_batch ->
    # snb_render_batch_fwd / bwd, csrc/render_batch.cu; the batched refine losses).  --per-object keeps round 1's path: one fused
    # render per object, the objects alternating over `--streams` CUDA streams.
    main_stream = torch.cuda.current_stream(dev)
    streams = [torch.cuda.Stream(device=dev) for _ in range(max(1, args.streams))] if (args.streams > 1 and not batched) else [main_stream]

    def fork():
        if len(streams) > 1:
            for st_ in streams:
                st_.wait_stream(main_stream)

    def join():
        if len(streams) > 1:
            for st_ in streams:
                main_stream.wait_stream(st_)

    wlhs, rois = [o["wlh"] for o in objs], [o["roi"] for o in objs]
    if batched:
        batch = R.make_batch(dev, torch.stack([o["img"] for o in objs]), torch.stack([o["mask_occ"] for o in objs]), wlhs,
                             torch.stack([o["K"] for o in objs]), rois, IM_SZ)
        cams = torch.stack([o["cam_pose"] for o in objs]).to(dev).requires_grad_()
        shps = torch.cat([o["shapecode"] for o in objs]).to(dev).requires_grad_()
        texs = torch.cat([o["texturecode"] for o in objs]).to(dev).requires_grad_()
        ones_b = torch.ones(N_OBJ, device=dev)
        # pinned host copies for `e2e`: one buffer per input kind for the whole batch
        h_img = torch.stack([o["img"] for o in objs]).pin_memory()
        h_mask = torch.stack([o["mask_occ"] for o in objs]).pin_memory()
        h_cam = torch.stack([o["cam_pose"] for o in objs]).pin_memory()
        h_K = torch.stack([o["K"] for o in objs]).pin_memory()
        h_shp = torch.cat([o["shapecode"] for o in objs]).pin_memory()
        h_tex = torch.cat([o["texturecode"] for o in objs]).pin_memory()

    last = {}   # what the latest step_resident() handed its caller (written by --dump-outputs)

    def step_resident():
        """One pass over the batch through the public API with every input already resident in HBM; the losses and their backward
        to the poses + latents close the step."""
        if batched:
            cams.grad = shps.grad = texs.grad = None
            rgb, dep, acc = R.render_batch(model, batch, cams, shps, texs, fused_sampler=args.fused_sampler)
            loss, parts = snb.losses.refine_loss_batch(rgb, acc, batch.rgb_tgt, batch.occ_pixels, 0.1)
            loss.backward(gradient=ones_b)     # every object's own loss, upstream gradient 1 each
            last.update(zip(OUTPUTS, (rgb, dep, acc, loss, cams.grad, shps.grad, texs.grad)))
            return parts
        fork()
        outs = []
        for i, d in enumerate(dobjs):
            with torch.cuda.stream(streams[i % len(streams)]):
                d["cam"].grad = d["shp"].grad = d["tex"].grad = None
                rgb, dep, acc, tgt, occ = R.render_rays(model, dev, d["img"], d["mask"], d["cam"], d["wlh"], d["K"], d["roi"], d["shp"],
                                                        d["tex"], im_sz=IM_SZ)
                loss = snb.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0]
                loss.backward()
                outs.append((rgb, dep, acc, loss, d["cam"].grad, d["shp"].grad, d["tex"].grad))
        join()
        last.update(zip(OUTPUTS, (list(o) for o in zip(*outs))))
        return loss

    # pinned result buffers: per object the loss (1) + d cam_pose (12) + d shapecode (256) + d texturecode (256)
    res_host = torch.empty(N_OBJ, 1 + 12 + 512, dtype=torch.float32).pin_memory()

    # e2e, batched path: renderer.GraphedBatchStep -- the step's H2D copies from the pinned host buffers, the batched render, the
    # losses, their backward and the D2H copy of the result replayed as ONE CUDA graph per step (--eager-e2e: the same step issued
    # call by call through render_rays_batch, as round 2's earlier lines were measured)
    stepper = None
    if batched and not args.eager_e2e:
        stepper = snb.renderer.GraphedBatchStep(R, model, dev, h_img, h_mask, h_cam, wlhs, h_K, rois, h_shp, h_tex, im_sz=IM_SZ, loss_occ_coef=0.1)

    def step_e2e():
        if stepper is not None:
            res = stepper.run()
            torch.cuda.synchronize()     # the step's losses and gradients are on the host when the step ends
            return float(res[:, 0].sum().item())
        if batched:
            # H2D of the step's inputs from pinned memory (crops, masks, poses, intrinsics, codes), the drop-in call, D2H of the result
            cam = h_cam.to(dev, non_blocking=True).requires_grad_()
            shp = h_shp.to(dev, non_blocking=True).requires_grad_()
            tex = h_tex.to(dev, non_blocking=True).requires_grad_()
            rgb, dep, acc, tgt, occ = R.render_rays_batch(model, dev, h_img, h_mask, cam, wlhs, h_K, rois, shp, tex, im_sz=IM_SZ)
            loss, parts = snb.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)
            loss.backward(gradient=ones_b)
            res_host.copy_(torch.cat([parts[:, :1], cam.grad.reshape(N_OBJ, 12), shp.grad, tex.grad], 1), non_blocking=True)
            torch.cuda.synchronize()
            return float(res_host[:, 0].sum().item())
        fork()
        for i, h in enumerate(hobjs):
            with torch.cuda.stream(streams[i % len(streams)]):
                cam = h["cam"].to(dev, non_blocking=True).requires_grad_()
                shp = h["shp"].to(dev, non_blocking=True).requires_grad_()
                tex = h["tex"].to(dev, non_blocking=True).requires_grad_()
                K = h["K"].to(dev, non_blocking=True)
                rgb, dep, acc, tgt, occ = R.render_rays(model, dev, h["img"], h["mask"], cam, h["wlh"], K, h["roi"], shp, tex, im_sz=IM_SZ)
                loss = snb.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0]
                loss.backward()
                # D2H read of the step's result: the loss and the gradients the refine loop consumes, into pinned memory
                res_host[i].copy_(torch.cat([loss.detach().reshape(1), cam.grad.reshape(-1), shp.grad.reshape(-1), tex.grad.reshape(-1)]),
                                  non_blocking=True)
        join()
        torch.cuda.synchronize()   # every object's result is on the host when the step ends
        return float(res_host[:, 0].sum().item())

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, **kw):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn(**kw)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        barrier()
        return ms

    for _ in range(max(args.warmup, 3)):
        step_resident()
    # the stratified-sampling jitter comes from the device generator: seeded here, the timed steps see the same jitter in every run
    # with the same --steps, whatever ran before them
    torch.cuda.manual_seed(0)
    launches0 = lib.snb_launch_count()
    with ClockSampler(local) as clk:
        ms_total = timed(step_resident, args.steps)
    launches = lib.snb_launch_count() - launches0
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    # Kernel-only pass for the roofline: the SAME step on ONE stream with CUDA events on the launch stream around the tcgen05
    # kernels alone.  (With several streams an event pair also spans the time a decoder kernel queues behind another stream's
    # decoder kernel -- the SMs hold one decoder CTA each -- so the multi-stream pass above is timed without them.)
    import ctypes
    all_streams = list(streams)
    streams[:] = [main_stream]
    step_resident()
    hnd = model._handle(dev).h
    lib.snb_kernel_timing_enable(hnd, 1)
    ms_single = timed(step_resident, args.steps)
    kern = {}
    for which, name in ((0, "fwd"), (1, "bwd")):
        buf = (ctypes.c_float * 4096)()
        n = lib.snb_kernel_timing_read(hnd, which, buf, 4096)
        kern[name] = [buf[i] for i in range(n)]
    lib.snb_kernel_timing_enable(hnd, 0)
    streams[:] = all_streams
    for _ in range(2):
        step_e2e()
    with ClockSampler(local) as clk2:
        ms_e2e = timed(step_e2e, args.steps)

    rays_per_step = N_OBJ * n_rays * world
    value = rays_per_step * args.steps / (ms_total / 1e3)
    e2e_value = rays_per_step * args.steps / (ms_e2e / 1e3)
    h2d = N_OBJ * (IM_SZ * IM_SZ * 3 * 4 + IM_SZ * IM_SZ * 4 + 12 * 4 + 9 * 4 + 2 * 256 * 4)
    d2h = N_OBJ * (1 + 12 + 512) * 4

    # roofline of the dominant kernel: the decoder MLP (tensor-pipe bound), from CUDA events recorded around the C-ABI
    # decoder calls inside the timed region (they bracket the tcgen05 kernel plus ~10 us of per-object latent GEMMs)
    pk = peaks()
    # Rows the decoder really executes (SURVEY 8d, accounting rule for miss rays): the fused bf16 render runs S rows per ray that
    # hits the box and ONE row per miss ray (csrc/compact.cu), padded to the 128-row tile; rays/s still counts every ray.
    rows_full = n_rays * N_SAMPLES
    rows_exec = []
    with torch.no_grad():
        for d in dobjs:
            ro, vd = snb.utils.get_rays(d["K"], d["cam"], d["roi"], uv_steps=[IM_SZ, IM_SZ])
            hit = R.prepare_sampled_rays(ro, vd, d["wlh"])[3]
            nh = int(hit.sum().item())
            compacted = (args.precision == "bf16" or fp32_tc) and os.environ.get("SNB_NO_COMPACT", "0") in ("", "0")
            pad = 256 if batched else 128
            rows_exec.append(-(-(nh * N_SAMPLES + (n_rays - nh)) // pad) * pad if compacted else rows_full)
            d["hit_fraction"] = nh / n_rays
    hit_fraction = float(np.mean([d["hit_fraction"] for d in dobjs]))
    rows = float(np.sum(rows_exec)) if batched else float(np.mean(rows_exec))   # one launch renders all objects in the batched path
    flop_per_launch = 2.0 * MAC_PER_SAMPLE * rows
    roof = {}
    for which in ("fwd", "bwd"):
        ts = kern.get(which) or []
        if ts:   # per-object path: launches cycle through the objects in order (pair every duration with its object's executed rows)
            per_launch = [rows] * len(ts) if batched else [rows_exec[i % N_OBJ] for i in range(len(ts))]
            tf = [2.0 * MAC_PER_SAMPLE * r_ / (t / 1e3) / 1e12 for r_, t in zip(per_launch, ts)]
            avg = float(np.mean(ts))
            roof[which] = dict(ms=avg, tflops=float(np.sum([2.0 * MAC_PER_SAMPLE * r_ for r_ in per_launch]) / (np.sum(ts) / 1e3) / 1e12),
                               n=len(ts), total_ms=float(np.sum(ts)), tflops_min=float(min(tf)), tflops_max=float(max(tf)))
    dom = max(roof, key=lambda k: roof[k]["total_ms"]) if roof else None
    # fp32 on the tensor cores issues three fp16 MMAs per product: its ceiling in fp32-equivalent FLOP/s is a third of the MMA peak
    peak = pk["tf_sustained"] if args.precision == "bf16" else (round(pk["tf_sustained"] / 3, 1) if fp32_tc else None)
    roofline = None
    traffic = None
    try:   # DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture (scaled by samples per launch)
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))
        k = tj["tc2_%s_kernel" % dom]
        traffic = int((k["dram_read_bytes"] + k["dram_write_bytes"]) * rows / tj["samples_per_captured_launch"])   # scaled to the executed rows
    except Exception:
        traffic = None
    if dom:
        roofline = {"bound": "tensor", "kernel": "tc2_%s_kernel" % dom if args.precision == "bf16" else
                    ("tc_%s_kernel<split> (SNB_PREC_FP32_TC: two fp16 parts per operand, three tcgen05 MMAs per product)" % dom if fp32_tc else "sgemm_kernel (fp32 SIMT)"),
                    "achieved": round(roof[dom]["tflops"], 2), "peak": peak, "unit": "TFLOP/s",
                    "frac": round(roof[dom]["tflops"] / peak, 4) if peak else None,
                    "frac_vs_burst_peak": round(roof[dom]["tflops"] / (pk["tf_burst"] / (3 if fp32_tc else 1)), 4) if (args.precision == "bf16" or fp32_tc) else None, "traffic": traffic if args.precision == "bf16" else None,
                    "peak_source": pk["source"] + (", sustained bf16" if not fp32_tc else ", sustained bf16 / 3 (three MMAs per fp32-grade product)"), "flop_per_launch": flop_per_launch,
                    "rows_executed_per_launch": rows, "rows_reference_semantics": rows_full, "hit_fraction": round(hit_fraction, 4),
                    "accounting": "achieved = 2 x 449664 MAC x rows the decoder EXECUTED (S per hit ray + 1 per miss ray, 128-row padded) / kernel time; "
                                  "value (rays/s) counts all rays, as the reference pushes all N x S rows through its MLP",
                    "avg_launch_ms": round(roof[dom]["ms"], 4),
                    "other": {k: {"ms": round(v["ms"], 4), "tflops": round(v["tflops"], 2)} for k, v in roof.items()},
                    "mlp_share_of_step": round(sum(v["total_ms"] for v in roof.values()) / (ms_single if batched else ms_total), 4),
                    "mlp_share_of_single_stream_step": round(sum(v["total_ms"] for v in roof.values()) / ms_single, 4),
                    "single_stream_ms_per_step": round(ms_single / args.steps, 3),
                    "timed": "CUDA events on the launch stream around the kernel alone, over a timed pass of the same step on ONE "
                             "stream (K steps, right after the multi-stream pass `value` comes from: there an event pair would also "
                             "span the kernel's wait behind another stream's decoder kernel)" if kern.get("fwd") else
                             "CUDA events around the decoder C-ABI call"}

    # secondary roofline, HBM-bound: the compositing kernels on one step's worth of rays (16 x 16384 rays x 64 samples: 335 MB in,
    # larger than L2), forward and backward, CUDA events around the C-ABI calls on the launch stream
    comp = None
    if rank == 0 and not args.no_extras:
        try:
            nr = N_OBJ * n_rays
            g = torch.Generator().manual_seed(0)
            sg = (torch.rand(nr, N_SAMPLES, generator=g) * 4 - 1).to(dev)
            cg = torch.rand(nr, N_SAMPLES, 3, generator=g).to(dev)
            zg = (torch.rand(nr, N_SAMPLES, generator=g).sort(-1).values + 0.5).to(dev)
            o3, o1, o2 = torch.empty(nr, 3, device=dev), torch.empty(nr, device=dev), torch.empty(nr, device=dev)
            go3, go1, go2 = torch.rand(nr, 3, device=dev), torch.rand(nr, device=dev), torch.rand(nr, device=dev)
            gsg, gcg, gzg = torch.empty_like(sg), torch.empty_like(cg), torch.empty_like(zg)
            P, stp = _lib.ptr, _lib.stream_ptr()

            def cf():
                _lib.check(lib.snb_composite_fwd(P(sg), P(cg), P(zg), 1, nr, N_SAMPLES, 3, P(o3), P(o1), P(o2), stp), "composite_fwd")

            def cb():
                _lib.check(lib.snb_composite_bwd(P(sg), P(cg), P(zg), 1, nr, N_SAMPLES, 3, P(go3), P(go1), P(go2), P(gsg), P(gcg), P(gzg), stp),
                           "composite_bwd")
            res = {}
            for name, fn, nbytes in (("fwd", cf, nr * (20 * N_SAMPLES + 20)), ("bwd", cb, nr * (40 * N_SAMPLES + 20))):
                for _ in range(3):
                    fn()
                ts = []
                for _ in range(7):
                    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a0.record(); fn(); a1.record()
                    torch.cuda.synchronize()
                    ts.append(a0.elapsed_time(a1))
                t = float(np.median(ts))
                res[name] = {"ms": round(t, 4), "gbs": round(nbytes / t / 1e6, 1), "frac": round(nbytes / t / 1e6 / peaks()["hbm"], 4),
                             "algorithmic_bytes": int(nbytes)}
            tot_b = res["fwd"]["algorithmic_bytes"] + res["bwd"]["algorithmic_bytes"]
            tot_t = res["fwd"]["ms"] + res["bwd"]["ms"]
            comp = {"bound": "hbm", "kernel": "composite_fwd4_kernel + composite_bwd4_kernel", "achieved": round(tot_b / tot_t / 1e6, 1),
                    "peak": peaks()["hbm"], "unit": "GB/s", "frac": round(tot_b / tot_t / 1e6 / peaks()["hbm"], 4), "fwd": res["fwd"], "bwd": res["bwd"],
                    "rays": nr, "samples_per_ray": N_SAMPLES, "bytes_per_ray": "fwd 20 S + 20, bwd 40 S + 20 (SURVEY 8d)",
                    "timed": "CUDA events around the C-ABI call, median of 7, inputs 335 MB (> L2)"}
            del sg, cg, zg, gsg, gcg, gzg
        except Exception as exc:   # never lose the headline line over the secondary measurement
            comp = {"error": str(exc)}
    # the metric's second half, "ms per refine iteration" (config C3 shape: one object, 32x32 rays x 64 samples, pose + codes
    # optimised with AdamW): refine.ObjectRefiner, one CUDA graph per iteration, 50 iterations, CUDA events
    refine_it = None
    if rank == 0 and not args.no_extras:
        try:
            import numpy as _np
            sup = snb.SUPNeRF(3, 1, 3, 3, 256)
            sup.load_state_dict(sd)
            sup = sup.to(dev)
            sup.precision = args.precision
            sup.requires_grad_(False)

            def refiner_uncaptured(k, max_iters):
                return refiner_for(k, max_iters, capture=False)

            def refiner_for(k, max_iters, capture=True):
                o = make_objects(300 + k, 1, 32)[0]
                c2o = o["cam_pose"]
                r_obj = c2o[:, :3].t().contiguous().double()
                t_obj = -(r_obj.float() @ c2o[:, 3:]).reshape(3)
                ang = torch.acos(((torch.trace(r_obj) - 1) / 2).clamp(-1, 1))
                w = torch.stack([r_obj[2, 1] - r_obj[1, 2], r_obj[0, 2] - r_obj[2, 0], r_obj[1, 0] - r_obj[0, 1]])
                rot_vec = (w / (2 * torch.sin(ang).clamp_min(1e-12)) * ang).float()
                rs = _np.random.RandomState(300 + k)   # 64 "lidar" pixels of the crop: their no-grad depth render is part of every iteration
                lidar = (rs.randint(0, o["img"].shape[1], 64), rs.randint(0, o["img"].shape[0], 64))
                r_ = snb.refine.ObjectRefiner(sup, dev, o["img"].to(dev), o["mask_occ"].to(dev), o["K"], o["roi"],
                                              _np.linalg.norm(o["wlh"]).astype(_np.float32), o["shapecode"], o["texturecode"], rot_vec,
                                              t_obj, n_samples=N_SAMPLES, im_sz=32, max_iters=max_iters, lidar_xy=lidar)
                return r_.capture() if capture else r_

            ref = refiner_for(0, 60)
            ref.run(5)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            last = ref.run(50)
            a1.record()
            torch.cuda.synchronize()
            refine_it = {"ms_per_refine_iteration": round(a0.elapsed_time(a1) / 50, 4), "iterations": 50,
                         "config": "configs[2] shape: one object, 32x32 rays x %d samples, AdamW on pose + shape/texture codes, "
                                   "supnerf_b200.refine.ObjectRefiner (one CUDA graph per iteration), INCLUDING the per-iteration evaluation of "
                                   "optimizer_nuscenes.py:740-769 (PSNR loss over the object mask + no-grad depth render of 64 lidar pixels)" % N_SAMPLES,
                         "loss_after": round(float(last[0]), 5)}
            # configs[2] gives every GPU 4 objects: refined side by side (refine.run_objects, one stream per object)
            refs = [refiner_for(k, 60) for k in range(4)]
            snb.refine.run_objects(refs, 5, 4)
            torch.cuda.synchronize()
            a0.record()
            snb.refine.run_objects(refs, 50, 4)
            a1.record()
            torch.cuda.synchronize()
            refine_it["four_objects_side_by_side"] = {
                "ms_per_refine_iteration": round(a0.elapsed_time(a1) / (4 * 50), 4), "objects": 4, "iterations": 50, "cuda_streams": 4,
                "note": "per object-iteration: elapsed / (4 objects x 50 iterations) (configs[2]: 4 objects per GPU), refine.run_objects"}
            # ... and from ONE CUDA graph per iteration whose four branches the device schedules (refine.ObjectGroup)
            grp = snb.refine.ObjectGroup([refiner_uncaptured(k, 60) for k in range(4)]).capture()
            grp.run(5)
            torch.cuda.synchronize()
            a0.record()
            grp.run(50)
            a1.record()
            torch.cuda.synchronize()
            refine_it["four_objects_one_graph"] = {
                "ms_per_refine_iteration": round(a0.elapsed_time(a1) / (4 * 50), 4), "objects": 4, "iterations": 50,
                "note": "refine.ObjectGroup: the 4 objects' iterations forked / joined inside one captured graph, one graph launch per iteration"}
            # ... and as ONE launch set per iteration for all objects (refine.BatchRefiner: batched pose map, render, losses, AdamW)
            for nb in (1, 4, 16):
                bat = snb.refine.BatchRefiner([refiner_uncaptured(k, 60) for k in range(nb)]).capture()
                bat.run(5)
                torch.cuda.synchronize()
                a0.record()
                lastb = bat.run(50)
                a1.record()
                torch.cuda.synchronize()
                refine_it["%d_object%s_one_launch_set" % (nb, "" if nb == 1 else "s")] = {
                    "ms_per_refine_iteration": round(a0.elapsed_time(a1) / (nb * 50), 4), "objects": nb, "iterations": 50,
                    "ms_per_batched_iteration": round(a0.elapsed_time(a1) / 50, 4), "loss_after_obj0": round(float(lastb[0, 0]), 5),
                    "note": "refine.BatchRefiner: every stage of the iteration (incl. the lidar-pixel evaluation) once over all objects, "
                            "one captured graph; per object-iteration = elapsed / (objects x 50)"}
            # the same iteration in fp32 (1e-5 parity) mode: the split-precision tensor-core decoder, since no weight takes a gradient
            if args.precision == "bf16":
                sup.precision = "fp32"
                try:
                    r32 = refiner_for(0, 60)
                    r32.run(5)
                    torch.cuda.synchronize()
                    a0.record()
                    last32 = r32.run(50)
                    a1.record()
                    torch.cuda.synchronize()
                    refine_it["fp32_mode"] = {"ms_per_refine_iteration": round(a0.elapsed_time(a1) / 50, 4), "iterations": 50,
                                              "loss_after": round(float(last32[0]), 5),
                                              "note": "one object, precision='fp32' (SNB_PREC_FP32_TC decoder kernels), one CUDA graph per iteration"}
                finally:
                    sup.precision = args.precision
        except Exception as exc:
            refine_it = dict(refine_it or {}, error=str(exc))
    # the collective-bearing modes of the north star (configs[3], configs[4]): run at every N (N = 1 anchors the strong-scaling curve)
    modes = {}
    if not args.skip_modes:
        for key, fn in (("ray_sharded_c4", run_c4), ("dp_train_c5", run_c5)):
            try:
                modes[key] = fn(snb, dev, rank, world, args.steps, args.warmup, args.precision)
            except Exception as exc:   # never lose the headline line over a secondary mode
                import traceback
                traceback.print_exc()
                modes[key] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    # the CPU arm is timed on rank 0 at N = 1 only (at N > 1 the other ranks' processes share the host cores)
    # secondary measurements in child processes (N = 1 only): (a) the same step WITHOUT miss-ray compaction (SNB_NO_COMPACT=1: every
    # one of the N x S rows goes through the decoder, the reference's semantics row for row), (b) the fp32 (1e-5 parity) mode on the
    # split-precision tensor-core kernels (SNB_PREC_FP32_TC), (c) the same mode on the FFMA kernels (what weight training uses)
    extras = {}
    if world == 1 and not args.no_extras:
        for key, extra_args, env_add in (("dense_rows_no_compaction", ["--per-object", "--precision", "bf16"], {"SNB_NO_COMPACT": "1"}),
                                         ("fp32_parity_mode", ["--precision", "fp32"], {}),
                                         ("fp32_parity_mode_ffma", ["--per-object", "--precision", "fp32"], {"SNB_FP32_SIMT": "1"})):
            try:
                env = dict(os.environ, **env_add)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--skip-modes", "--no-extras", "--steps", "3", "--warmup", "3"] + extra_args,
                                   capture_output=True, text=True, timeout=420, env=env)
                sub = json.loads(r.stdout.strip().splitlines()[-1])
                extras[key] = {"value": sub["value"], "unit": "rays/s", "ms_per_step": sub["ms_per_step"], "e2e": sub["e2e"]["value"],
                               "precision": sub["config"]["precision"], "launch_sets": sub["config"].get("launch_sets"),
                               "decoder_tflops": (sub.get("roofline") or {}).get("other"), "decoder_kernel": (sub.get("roofline") or {}).get("kernel"),
                               "steps": sub["steps"]}
            except Exception as exc:   # noqa: BLE001
                extras[key] = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
    cpu = cpu_baseline(steps=3, warmup=1) if (world == 1 and not args.no_extras) else None
    eager = gpu_eager_baseline(dev) if (world == 1 and not args.no_extras) else None
    line = {"metric": METRIC, "value": round(value, 1), "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "objects_per_gpu": N_OBJ, "rays_per_object": n_rays, "samples_per_ray": N_SAMPLES, "weights": "frozen (refine mode)",
                       "grads": "cam_pose, shapecode, texturecode", "parallelism": "object-parallel x%d, no collective; every rank renders the same 16-object set" % world, "cuda_streams_per_gpu": len(streams),
                       "launch_sets": "one batched launch set for the 16 objects (snb_render_batch_fwd/bwd)" if batched else "one fused render per object",
                       "l2": "working set larger than L2 (126 MB): a step executes ~7 M decoder rows; per row 28 B of sample coordinates + z, 16 B of decoder outputs, as much again of gradients, and 224 B of ReLU mask bits (7 mask slots x 32 B) written by the forward and read by the backward: ~2 GB through HBM per step",
                       "hit_fraction": round(hit_fraction, 4),
                       "precision": args.precision,
                       "decoder_arithmetic": "bf16 x bf16 -> fp32 (tcgen05)" if args.precision == "bf16" else
                                             ("fp32-grade: fp16 (hi, lo) operand pairs, 3 tcgen05 MMAs per product -> fp32" if fp32_tc else "fp32 FFMA")},
            "e2e": {"value": round(e2e_value, 1), "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(ms_e2e / args.steps, 3),
                    "api": ("renderer.GraphedBatchStep.run(): pinned host inputs -> H2D, render_batch, refine_loss_batch, backward, D2H of the losses and "
                            "gradients into pinned memory, one CUDA graph launch per step, torch.cuda.synchronize() after every step") if stepper is not None
                           else "render_rays_batch / render_rays + refine losses + backward call by call, synchronize after every step"},
            "roofline_compositing": comp, "refine_iteration": refine_it, "gpu_launches": int(launches), "clocks": dict(clk.summary(), e2e_region=clk2.summary()), "roofline": roofline, "cpu_baseline": cpu, "gpu_eager_baseline": eager}
    line.update(extras)
    line.update(modes)
    if modes:
        line["multi_gpu_parity"] = "pass" if all(m.get("multi_gpu_parity", "pass") == "pass" and "error" not in m for m in modes.values()) else "FAIL"
    print(json.dumps(line), file=JSON_OUT, flush=True)


# ----------------------------------------------------------------------------------------------------- collective-bearing modes
def _maxr(x, dev, world, op="max"):
    """max (or min) over ranks of a python float / list of floats."""
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor(x if isinstance(x, (list, tuple)) else [x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.MIN)
    out = [float(v) for v in t.tolist()]
    return out if isinstance(x, (list, tuple)) else out[0]


def run_c4(snb, dev, rank, world, steps, warmup, precision):
    """configs[3]: ONE 512x512 object, 128 samples per ray, ray-sharded over the launched ranks (interleaved 128-ray tiles), weights /
    pose / codes replicated, ONE NCCL all-reduce of [d cam_pose | d shapecode | d texturecode | loss] (525 floats) per step.  STRONG
    scaling: total work fixed.  Self-checks what tests/test_gpu_multi.py asserts, on this very run, before timing."""
    import torch.distributed as dist
    from supnerf_b200 import parallel, synthetic
    IM, S = 512, 128
    LAYOUT = "strided"   # ray i on rank i % G: balanced hit counts (128-ray tiles left the ranks 15 % apart, profiles/r2_c4_layouts.md)
    obj = synthetic.synthetic_object(4, im_sz=IM)
    sd = synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=4)
    m = snb.SUPNeRF(3, 1, 3, 3, 256)
    m.load_state_dict(sd)
    m = m.to(dev)
    m.precision = precision
    m.requires_grad_(False)
    R = snb.renderer.NeRFRenderer(n_samples=S)
    shp0, tex0 = synthetic.synthetic_latents(4, 1)
    img, mask, K = obj["img"].to(dev), obj["mask_occ"].to(dev), obj["K"].to(dev)

    def leaves():
        return obj["cam_pose"].to(dev).requires_grad_(), shp0.to(dev).requires_grad_(), tex0.to(dev).requires_grad_()

    # the gradient all-reduce goes through the C ABI (snb_allreduce_grads) on this process' own NCCL communicator
    comm = parallel.NcclComm(dev) if world > 1 else None
    shard = parallel.RayShard(R, m, dev, img, mask, obj["wlh"], K, obj["roi"], IM, rank=rank, world=world, layout=LAYOUT, comm=comm)
    whole = parallel.RayShard(R, m, dev, img, mask, obj["wlh"], K, obj["roi"], IM, rank=0, world=1, layout=LAYOUT, group=None)
    # ---- parity, on this run: the sharded step against the SAME step on one rank (every rank renders the whole object once)
    cam, shp, tex = leaves()
    loss_s, rgb_s, _, _ = shard.step(cam, shp, tex, seed=1234)
    g_sharded = torch.cat([cam.grad.reshape(-1), shp.grad.reshape(-1), tex.grad.reshape(-1)]).clone()
    cam1, shp1, tex1 = leaves()
    # one-rank reference: no collective (world 1 => allreduce_grads reduces over nothing)
    from supnerf_b200 import losses, ops
    jit = ops.jitter_fill(1234, IM * IM, S, dev)
    rgb_1, dep_1, acc_1 = R._render_fused(m, dev, whole.px, whole.py, K, cam1, obj["wlh"], shp1, tex1, jitter=jit)
    part = losses.refine_loss(rgb_1, acc_1, whole.rgb_tgt, whole.occ, 0.1, den=whole.den)[0]
    part.backward()
    g_one = torch.cat([cam1.grad.reshape(-1), shp1.grad.reshape(-1), tex1.grad.reshape(-1)])
    full = parallel.gather_rays(rgb_s.detach(), IM * IM, S, layout=LAYOUT) if world > 1 else rgb_s.detach()

    def rel(a, b):
        return float((a.double() - b.double()).abs().max() / b.double().abs().max())
    checks = {"loss_rel_err_vs_1rank": abs(float(loss_s) - float(part)) / abs(float(part)),
              "gathered_image_bit_identical": bool(torch.equal(full, rgb_1.detach())),
              "g_pose_rel_err_vs_1rank": rel(g_sharded[:12], g_one[:12]), "g_shape_rel_err_vs_1rank": rel(g_sharded[12:268], g_one[12:268]),
              "g_texture_rel_err_vs_1rank": rel(g_sharded[268:], g_one[268:])}
    if world > 1:
        gs = [torch.empty_like(g_sharded) for _ in range(world)]
        dist.all_gather(gs, g_sharded)
        checks["gradients_bit_identical_across_ranks"] = bool(all(torch.equal(gs[0], g) for g in gs[1:]))
    else:
        checks["gradients_bit_identical_across_ranks"] = True
    tol_g = 2e-2 if precision == "bf16" else 1e-3
    ok = (checks["loss_rel_err_vs_1rank"] <= 1e-5 and checks["gathered_image_bit_identical"] and checks["gradients_bit_identical_across_ranks"]
          and checks["g_shape_rel_err_vs_1rank"] <= tol_g and checks["g_texture_rel_err_vs_1rank"] <= tol_g and checks["g_pose_rel_err_vs_1rank"] <= tol_g)
    ok = bool(_maxr(0.0 if ok else 1.0, dev, world) == 0.0)
    del rgb_1, dep_1, acc_1, jit, full

    # ---- timing: K steps, phases marked with CUDA events on the launch stream
    cam, shp, tex = leaves()
    names = ("jitter", "forward", "backward", "allreduce")

    def timed(sh, k, record):
        evs = []
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(k):
            row = [torch.cuda.Event(enable_timing=True)]
            row[0].record()

            def mark(name, row=row):
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                row.append(e)
            loss = sh.step(cam, shp, tex, seed=1000 + i, events=mark if record else None)[0]
            evs.append(row)
        t1 = torch.cuda.Event(enable_timing=True)
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / k
        phases = None
        if record:
            phases = [float(np.mean([r[j].elapsed_time(r[j + 1]) for r in evs])) for j in range(len(names))]
        return ms, phases, float(loss)

    for _ in range(max(warmup, 3)):
        shard.step(cam, shp, tex, seed=1)
    ms_plain, _, loss = timed(shard, steps, False)          # the number: no per-phase events inside
    ms, phases, _ = timed(shard, steps, True)
    ms_max = _maxr(ms_plain, dev, world)
    ph_max = _maxr(phases, dev, world)
    ph_min = _maxr(phases, dev, world, "min")
    # one-GPU time of the same step IN THIS RUN (rank 0 alone renders the whole object; the other ranks wait)
    ms_one = None
    if world > 1:
        if rank == 0:
            for _ in range(2):
                whole.step(cam, shp, tex, seed=1)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for i in range(steps):
                whole.step(cam, shp, tex, seed=1000 + i)
            a1.record()
            torch.cuda.synchronize()
            ms_one = a0.elapsed_time(a1) / steps
        ms_one = _maxr(ms_one if ms_one is not None else 0.0, dev, world)
    n = IM * IM
    out = {"config": "configs[3]: one 512x512 object x 128 samples, ray-sharded x%d (ray i on rank i %% G), one all-reduce of 525 floats per step" % world,
           "scaling": "strong", "n_gpus": world, "ms_per_step": round(ms_max, 3), "rays_per_s": round(n / (ms_max / 1e3), 1),
           "precision": precision, "loss": loss,
           "one_gpu_ms_per_step_same_run": round(ms_one, 3) if ms_one else None,
           "efficiency_vs_one_gpu_same_run": round(ms_one / (world * ms_max), 4) if ms_one else None,
           "phases_ms_max_over_ranks": dict(zip(names, [round(v, 4) for v in ph_max])),
           "phases_ms_min_over_ranks": dict(zip(names, [round(v, 4) for v in ph_min])),
           "allreduce_us": round(1e3 * ph_max[3], 1),
           "phase_note": "CUDA events on the launch stream in a second timed pass of the same K steps; `allreduce` = torch.cat of the three "
                         "gradients + loss, snb_allreduce_grads (ncclAllReduce of 525 floats through the C ABI), views back; it also absorbs "
                         "the wait for the slowest rank's backward",
           "multi_gpu_parity": "pass" if ok else "FAIL", "parity_checks": checks}
    if comm is not None:
        comm.destroy()
    return out


def run_c5(snb, dev, rank, world, steps, warmup, precision):
    """configs[4]: the joint training step of trainer_unified_nuscenes.py:27-148 + :316-329 per GPU -- pose-estimator forward
    (ImgEncoder on (8,3,128,128) crops, bf16 channels-last cuDNN; direct corner regression; 3 pose-regress iterations), the render of
    8 objects x 1024 rays x 64 samples through the decoder with EVERY weight gradient (tcgen05 training mode), all losses, backward
    through both halves, data-parallel all-reduce of all 49 M gradients (196 MB) in 3 buckets overlapped with the encoder's
    backward, fused AdamW on weights + codes.  WEAK scaling: every rank its own 8 objects."""
    import torch.distributed as dist
    from supnerf_b200 import parallel, pose_estimator as pe, synthetic
    B, n, S = 8, 1024, N_SAMPLES
    g = torch.Generator().manual_seed(50 + rank)
    sd = dict(synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=5))
    m = snb.SUPNeRF(3, 1, 3, 3, 256)
    m.materialize_pose_estimator()
    sd.update(synthetic.pose_estimator_state(m.state_dict(), 5))
    m.load_state_dict(sd)
    m = m.to(dev).to(memory_format=torch.channels_last)
    m.precision = precision
    m.train()
    img = torch.rand(B, 3, 128, 128, generator=g).to(dev)
    xyz = ((torch.rand(B, n, S, 3, generator=g) - 0.5) * 1.2).to(dev)
    vd = torch.nn.functional.normalize(torch.randn(B, n, 1, 3, generator=g), dim=-1).repeat(1, 1, S, 1).to(dev)
    zv = (torch.rand(B, S, generator=g).sort(-1).values * 4 + 8).to(dev)
    tgt, occ = torch.rand(B, n, 3, generator=g).to(dev), torch.randint(-1, 2, (B, n, 1), generator=g).float().to(dev)
    objs = [synthetic.synthetic_object(500 + rank * B + i, im_sz=16) for i in range(B)]
    c2o = torch.stack([o["cam_pose"] for o in objs])
    R_o2c = c2o[:, :, :3].transpose(1, 2)
    obj_pose = torch.cat([R_o2c, -R_o2c @ c2o[:, :, 3:]], -1).contiguous().to(dev)
    wlh = torch.stack([torch.from_numpy(np.asarray(o["wlh"], dtype=np.float32)) for o in objs]).to(dev)
    K = torch.stack([o["K"] for o in objs]).to(dev)
    roi = torch.stack([torch.as_tensor(np.asarray(o["roi"]), dtype=torch.float32) for o in objs]).to(dev)
    tgt_uv = pe.view_points_batch(pe.corners_of_box_batch(obj_pose, wlh), K, normalize=True)[:, :2, :]
    src_pose = torch.cat([obj_pose[:, :, :3], obj_pose[:, :, 3:] * torch.tensor([1.03, 0.98, 1.05], device=dev).view(1, 3, 1)], -1)
    shp0, tex0 = synthetic.synthetic_latents(5 + rank, B)
    shp, tex = shp0.to(dev).requires_grad_(), tex0.to(dev).requires_grad_()
    hp = {"loss_pose_coef": 0.01, "loss_code_coef": 0.1, "loss_occ_coef": 0.1}
    enc = m.img_encoder
    trunk = [p_ for mod in (enc.conv1, enc.bn1, enc.layer1, enc.layer2, enc.layer3) for p_ in mod.parameters()]
    branches = [p_ for mod in (enc.layer4_shape, enc.layer4_texture, enc.layer4_pose) for p_ in mod.parameters()]
    seen = set(id(p_) for p_ in trunk + branches)
    early = [p_ for p_ in m.parameters() if id(p_) not in seen]          # decoder, pose head, encoder heads: ready first
    n_params = sum(p_.numel() for p_ in m.parameters())
    opt = torch.optim.AdamW([{"params": list(m.parameters()), "lr": 1e-4}, {"params": [shp, tex], "lr": 1e-3}], fused=True)
    # The library stages of the step (the cuDNN encoder, ~330 launches forward + backward; the three pose-regress iterations, ~600
    # small torch kernels) are launch-bound when issued eagerly (the eager step takes 21.6 ms on one B200, of which 2.5 ms is the
    # render): both are captured as CUDA graphs (forward and backward) with torch.cuda.make_graphed_callables; the render half is
    # the package's own kernels.  If a capture fails the stage stays eager (reported).
    graphed = {"encoder": False, "pose_regress": False}
    K_inv = torch.linalg.inv(K)
    img_cl = img.contiguous(memory_format=torch.channels_last)
    encode, regress3 = m.encode_img_fast, None
    if os.environ.get("SNB_C5_EAGER", "0") in ("", "0"):
        try:
            with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
                enc_g = torch.cuda.make_graphed_callables(enc, (img_cl,), num_warmup_iters=3)

            def encode(_img):
                with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
                    out = enc_g(img_cl)
                return tuple(t.float() for t in out) + (None,)
            graphed["encoder"] = True
        except Exception as exc:   # noqa: BLE001
            graphed["encoder_error"] = "%s: %s" % (type(exc).__name__, str(exc)[:200])
        try:
            r3 = pe.PoseRegress3(m)
            sample = (torch.randn(B, 256, device=dev, requires_grad=True), src_pose, tgt_uv, wlh, roi, K, K_inv)
            r3_g = torch.cuda.make_graphed_callables(r3, sample, num_warmup_iters=3)

            def regress3(posecode, src, tuv, wl, ro, K_):
                return r3_g(posecode, src, tuv, wl, ro, K_, K_inv)
            graphed["pose_regress"] = True
        except Exception as exc:   # noqa: BLE001
            graphed["pose_regress_error"] = "%s: %s" % (type(exc).__name__, str(exc)[:200])
            regress3 = None
    buckets = parallel.BucketedGradAllReduce([early, branches, trunk])

    def step(overlap=True):
        m.zero_grad(set_to_none=True)
        shp.grad = tex.grad = None
        losses_all, total, *_ = pe.joint_training_losses(m, hp, img, shp, tex, xyz, vd, zv, tgt, occ, src_pose, tgt_uv, roi, K, wlh, tgt_uv,
                                                         encode=encode, regress3=regress3)
        if overlap:
            total.backward()
            buckets.finish()
        else:                      # the same exchange as ONE flat all-reduce after the whole backward (no overlap)
            saved = buckets.world
            buckets.world = 1
            total.backward()
            buckets.finish()
            buckets.world = saved
            if world > 1:
                parallel.allreduce_weight_grads(m)
        opt.step()
        return total.detach()

    def timed(k, **kw):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(k):
            loss = step(**kw)
        a1.record()
        torch.cuda.synchronize()
        return _maxr(a0.elapsed_time(a1) / k, dev, world), float(loss)

    for _ in range(max(warmup, 3)):
        step(overlap=False)
    # default exchange: ONE flat all-reduce of all gradients after the backward.  The bucketed, hook-driven exchange on a side
    # stream (parallel.BucketedGradAllReduce) is timed beside it: with the encoder backward replayed as one CUDA graph its gradients
    # all arrive together, so only the decoder / head bucket can overlap, and the per-parameter hook bookkeeping costs more host
    # time than the 1.2 ms exchange could hide
    ms, loss = timed(steps, overlap=False)

    def weights_identical():
        torch.cuda.synchronize()
        probe = torch.cat([m.encoding_xyz[0].weight.reshape(-1)[:64], enc.conv1.weight.reshape(-1)[:64], enc.layer4_pose[2].conv2.weight.reshape(-1)[:64],
                           m.out_delta_layer.weight.reshape(-1)[:64]])
        gs = [torch.empty_like(probe) for _ in range(world)]
        dist.all_gather(gs, probe)
        return bool(all(torch.equal(gs[0], t) for t in gs[1:]))
    same_flat = weights_identical() if world > 1 else None
    ms_bucketed, ar, same_bucketed = None, {}, None
    if world > 1 and not (graphed["encoder"] or graphed["pose_regress"]):
        # the hook-driven bucketed exchange needs gradients that arrive layer by layer: only meaningful with the EAGER library stages
        # (SNB_C5_EAGER=1); with the encoder backward replayed as one CUDA graph all its gradients arrive together
        for _ in range(2):
            step(overlap=True)
        ms_bucketed, _ = timed(steps, overlap=True)
        ar = buckets.allreduce_ms()
        same_bucketed = weights_identical()
    # phase split on one rank's stream (second pass, events): encoder+pose forward | render forward | backward | optimizer
    # SURVEY 8f rank 3: the step's samples prepared on the device (utils.prepare_pixel_samples_batch) instead of by DataLoader workers
    prep = None
    if rank == 0:
        try:
            pobjs = [synthetic.synthetic_object(700 + i, im_sz=64) for i in range(B)]
            pargs = (dev, [o["img"] for o in pobjs], [o["mask_occ"] for o in pobjs], [o["cam_pose"] for o in pobjs],
                     [np.linalg.norm(o["wlh"]).astype(np.float32) for o in pobjs], [o["K"] for o in pobjs], [o["roi"] for o in pobjs], n, S, 1, 0)
            for _ in range(2):
                snb.utils.prepare_pixel_samples_batch(*pargs, im_sz=64)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(5):
                pxyz = snb.utils.prepare_pixel_samples_batch(*pargs, im_sz=64)[0]
            torch.cuda.synchronize()
            prep = {"ms_per_batch_host_plus_device": round((time.perf_counter() - t0) / 5 * 1e3, 3), "objects": B, "rays": n, "samples": S,
                    "bytes_over_pcie_here": int(B * (S * 4 + 2 * n * 4 + n * 16 + 21 * 4)), "bytes_over_pcie_reference_loader": int(B * (2 * n * S * 12 + S * 4 + n * 16)),
                    "what": "utils.prepare_pixel_samples (data_nuscenes.py:643-658) for the whole batch in one kernel on the device; bit-identical "
                            "to per-object calls (tests/test_gpu_parity.py)", "shape": list(pxyz.shape)}
        except Exception as exc:   # noqa: BLE001
            prep = {"error": "%s: %s" % (type(exc).__name__, str(exc)[:200])}
    finite = bool(np.isfinite(loss))
    flops_dec = 3 * 2 * MAC_PER_SAMPLE * B * n * S
    out = {"config": "configs[4]: joint training step per GPU: ImgEncoder (8,3,128,128) bf16 channels-last + pose regression x3 + render of "
                     "%d objects x %d rays x %d samples fwd/bwd with all weight gradients + AdamW; data-parallel x%d, %d parameters (%.0f MB of "
                     "gradients) all-reduced every step" % (B, n, S, world, n_params, n_params * 4 / 1e6),
           "scaling": "weak", "n_gpus": world, "ms_per_step": round(ms, 3), "rays_per_s": round(world * B * n / (ms / 1e3), 1),
           "decoder_tflops_per_gpu_if_step_were_decoder_only": round(flops_dec / (ms / 1e3) / 1e12, 1),
           "loss": loss, "loss_finite": finite, "precision": precision, "parameters": n_params, "cuda_graphed_library_stages": graphed,
           "device_side_sample_prep": prep,
           "exchange": "one flat all-reduce (sum) of all %d gradients after the backward, scaled by 1/G" % n_params if world > 1 else "none (1 GPU)",
           "ms_per_step_bucketed_overlap": round(ms_bucketed, 3) if ms_bucketed else None,
           "bucketed_allreduce_ms_by_bucket": {"early(decoder+heads)": round(ar.get(0, 0.0), 3), "layer4 branches": round(ar.get(1, 0.0), 3),
                                               "trunk": round(ar.get(2, 0.0), 3)} if ar else None,
           "overlap_gain_ms": round(ms - ms_bucketed, 3) if ms_bucketed else None,
           "multi_gpu_parity": "pass" if finite else "FAIL"}
    if world > 1:   # every rank must hold identical weights after training (same reduced gradients, same update)
        out["weights_bit_identical_across_ranks_after_training"] = same_flat
        if same_bucketed is not None:
            out["weights_bit_identical_after_bucketed_steps"] = same_bucketed
        if not same_flat or same_bucketed is False:
            out["multi_gpu_parity"] = "FAIL"
    buckets.remove()
    return out


# ----------------------------------------------------------------------------------------------------- reference arms
def load_reference():
    """The UNMODIFIED reference staged under baseline/_ref/ by baseline/install_ref.py (its renderer.py / utils.py / model_*.py,
    byte for byte; matplotlib, which utils.py imports for an off-path colour map, is stubbed).  None if it was not staged."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "renderer.py")):
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import install_ref
            if not install_ref.install(verbose=False):
                return None
        except Exception:
            return None
    import importlib
    import types
    sys.modules.setdefault("matplotlib", types.ModuleType("matplotlib"))
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import warnings
    warnings.filterwarnings("ignore")
    mods = {name: importlib.import_module(name) for name in ("renderer", "model_autorf")}
    mods["manifest"] = json.load(open(os.path.join(ref_dir, "MANIFEST.json")))["sha256"] if os.path.exists(os.path.join(ref_dir, "MANIFEST.json")) else None
    return mods


def reference_model(ref, device):
    """The reference's own AutoRFMix(3, 1, 256) module with the bench's weights (same state_dict keys: decoder entries only)."""
    from supnerf_b200 import synthetic
    sd = synthetic.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=0)
    m = ref["model_autorf"].AutoRFMix(shape_blocks=3, texture_blocks=1, latent_dim=256)
    res = m.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    m = m.to(device)
    m.requires_grad_(False)   # refine mode, as in the measured arm
    return m


def reference_step(ref, R, model, objs, device):
    """One pass over `objs` through the reference's NeRFRenderer.render_rays (renderer.py:117-167) + the refine losses
    (optimizer_nuscenes.py:729-736) + backward to pose and codes: the reference's stock code path, device = cpu or cuda."""
    total = 0.0
    for o in objs:
        cam = o["cam_pose"].to(device).requires_grad_()
        shp, tex = o["shapecode"].to(device).requires_grad_(), o["texturecode"].to(device).requires_grad_()
        rgb, dep, acc, tgt, occ = R.render_rays(model, device, o["img"], o["mask_occ"], cam, o["wlh"], o["K"], o["roi"], shp, tex, im_sz=IM_SZ)
        loss = refine_loss(rgb, acc, tgt, occ)
        loss.backward()
        total += float(loss.detach())
    return total


def cpu_render_step(oracle, sd, obj, jitter):
    cam = obj["cam_pose"].clone().requires_grad_()
    shp, tex = obj["shapecode"].clone().requires_grad_(), obj["texturecode"].clone().requires_grad_()
    im = obj["img"].shape[0]
    rgb, dep, acc, _ = oracle.render_rays_box(sd, obj["K"], cam, obj["wlh"], obj["roi"], im, N_SAMPLES, shp, tex, jitter)
    loss = refine_loss(rgb, acc, obj["img"].reshape(-1, 3), obj["mask_occ"].reshape(-1, 1))
    loss.backward()
    return loss


CPU_SAMPLE_OBJECTS = 1   # objects of the 16-object set one CPU step renders (1 object = 16 384 rays x 64 samples = 1 M decoder rows)


def cpu_baseline(steps, warmup):
    """The reference's CPU path on the host cores, all threads: `kind: reference` = the unmodified reference (baseline/_ref) through
    its own NeRFRenderer.render_rays on the first CPU_SAMPLE_OBJECTS objects of the SAME 16-object set at the same 128x128 rays x 64
    samples; `kind: port` (only if the reference was not staged) = the oracle port on one 64x64-ray object."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ref = load_reference()
    if ref is not None:
        model = reference_model(ref, "cpu")
        R = ref["renderer"].NeRFRenderer(n_samples=N_SAMPLES)
        objs = make_objects(100, N_OBJ, IM_SZ)[:CPU_SAMPLE_OBJECTS]
        torch.manual_seed(0)
        for _ in range(warmup):
            reference_step(ref, R, model, objs, "cpu")
        ts = []
        for _ in range(steps):
            t0 = time.perf_counter()
            reference_step(ref, R, model, objs, "cpu")
            ts.append(time.perf_counter() - t0)
        sec = float(np.median(ts))
        rays = len(objs) * IM_SZ * IM_SZ
        return {"value": round(rays / sec, 1), "unit": "rays/s", "cores": cores, "kind": "reference", "rays_per_step": rays, "s_per_step": round(sec, 3),
                "sample": "unmodified reference (baseline/_ref: renderer.NeRFRenderer.render_rays + model_autorf.AutoRFMix(3,1,256)), torch CPU fp32, "
                          "%d of the 16 objects of configs[1] per step (%dx%d rays x %d samples each), fwd+bwd to pose+codes, weights frozen, "
                          "%d steps (median %.2f s/step)" % (len(objs), IM_SZ, IM_SZ, N_SAMPLES, steps, sec),
                "reference_sha256": ref["manifest"]}
    from oracle import oracle
    im_sz = 64
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=0)
    obj = make_objects(100, 1, im_sz)[0]
    jitter = torch.rand(im_sz * im_sz, N_SAMPLES, generator=torch.Generator().manual_seed(0))
    for _ in range(warmup):
        cpu_render_step(oracle, sd, obj, jitter)
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        cpu_render_step(oracle, sd, obj, jitter)
        ts.append(time.perf_counter() - t0)
    sec = float(np.median(ts))
    return {"value": round(im_sz * im_sz / sec, 1), "unit": "rays/s", "cores": cores, "kind": "port", "rays_per_step": im_sz * im_sz, "s_per_step": round(sec, 3),
            "sample": "oracle port (reference not staged): 1 object, %dx%d rays x %d samples, fwd+bwd to pose+latents, weights frozen, %d steps (median %.2f s/step)"
                      % (im_sz, im_sz, N_SAMPLES, steps, sec)}


def gpu_eager_baseline(dev, steps=3, warmup=2):
    """The reference's own eager PyTorch path on the SAME B200 (SURVEY 8d / BASELINE.md section 4: "the real same-box bar"): the
    unmodified reference with device='cuda', fp32, TF32 off (torch default), weights frozen, the full 16-object step of configs[1]."""
    ref = load_reference()
    if ref is None:
        return {"unavailable": "reference not staged under baseline/_ref"}
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    model = reference_model(ref, dev)
    R = ref["renderer"].NeRFRenderer(n_samples=N_SAMPLES)
    objs = make_objects(100, N_OBJ, IM_SZ)
    for _ in range(warmup):
        reference_step(ref, R, model, objs, dev)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        reference_step(ref, R, model, objs, dev)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    del model
    torch.cuda.empty_cache()
    return {"value": round(N_OBJ * IM_SZ * IM_SZ / (ms / 1e3), 1), "unit": "rays/s", "ms_per_step": round(ms, 3), "steps": steps, "warmup": warmup,
            "kind": "reference", "device": torch.cuda.get_device_name(dev), "dtype": "f32 (allow_tf32 = False)",
            "what": "unmodified reference (baseline/_ref) NeRFRenderer.render_rays + refine losses + backward, device='cuda', eager PyTorch, "
                    "the same 16 objects x 128x128 rays x 64 samples per step, inputs as the reference takes them (host img / mask, .to(device) inside)",
            "peak_memory_gib": round(peak_gb, 2)}


def run_reference(args):
    if int(os.environ.get("RANK", 0)) != 0:
        return
    steps, warmup = args.steps, args.warmup
    t0 = time.perf_counter()
    cpu = cpu_baseline(steps=steps, warmup=warmup)
    wall = time.perf_counter() - t0
    line = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "rays/s", "n_gpus": int(os.environ.get("WORLD_SIZE", 1)),
            "steps": steps, "warmup": warmup, "ms_per_step": round(1e3 * cpu["s_per_step"], 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "objects_per_gpu": N_OBJ, "rays_per_object": IM_SZ * IM_SZ, "samples_per_ray": N_SAMPLES,
                       "weights": "frozen (refine mode)", "grads": "cam_pose, shapecode, texturecode",
                       "bounded_sample": cpu["sample"]},
            "cpu_baseline": cpu, "e2e": {"value": cpu["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": round(wall, 1)}
    print(json.dumps(line), file=JSON_OUT, flush=True)


JSON_OUT = sys.stdout


def main():
    # stdout carries exactly ONE JSON line: anything a library prints there (e.g. NCCL's version banner under NCCL_DEBUG=VERSION)
    # is diverted to stderr by pointing fd 1 at fd 2 and keeping a private handle on the real stdout for the result
    global JSON_OUT
    JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--eager-e2e", action="store_true", help="e2e through render_rays_batch call by call instead of renderer.GraphedBatchStep (one CUDA graph per step)")
    ap.add_argument("--per-object", dest="batched", action="store_false",
                    help="round 1's path: one fused render per object over --streams CUDA streams (default: all objects in one launch set)")
    ap.add_argument("--fused-sampler", action="store_true",
                    help="north-star kernel K1: the decoder's forward computes its rows' samples from the rays (default: a sampler kernel writes them)")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (dense rows, fp32 mode, CPU / eager-CUDA reference baselines)")
    ap.add_argument("--skip-modes", action="store_true", help="skip the configs[3] / configs[4] collective-bearing modes")
    ap.add_argument("--streams", type=int, default=3, help="CUDA streams the independent objects alternate over (1 = one stream)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rendered rgb / depth / acc, losses, pose and code gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
