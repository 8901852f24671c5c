#!/usr/bin/env python
"""Short, self-contained run of the bench workload: `--warmup` + `--steps` measured steps of `--objects` objects (128x128 rays x 64
samples each, fwd+bwd to pose + latents).  Prints the step time (CUDA events) and rays/s.
  --decoder bench       AutoRF-mix 3/1/256 (the bench decoder); autorfmix: AutoRFMix()'s class defaults, 5/5 blocks at W = latent_dim = 128
  --path unfused        per object: get_rays, prepare_sampled_rays, decoder, volume_render (one call each)
         per-object     per object: NeRFRenderer.render_rays (the fused per-object render)
         batched        every object in one NeRFRenderer.render_rays_batch launch set (configs[1] at --objects 16)
With SNB_FP32_SIMT=1 in the environment, fp32 mode runs the decoder on the FFMA back end."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import supnerf_b200 as snb  # noqa: E402
from oracle import oracle  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--objects", type=int, default=2)
ap.add_argument("--precision", default="bf16")
ap.add_argument("--im-sz", type=int, default=128)
ap.add_argument("--decoder", default="bench", choices=["bench", "autorfmix"])
ap.add_argument("--path", default="unfused", choices=["unfused", "per-object", "batched"])
ap.add_argument("--steps", type=int, default=1)
ap.add_argument("--warmup", type=int, default=1)
a = ap.parse_args()
dev = torch.device("cuda", 0)
if a.decoder == "bench":
    D = 256
    sd = oracle.init_codenerf_state(shape_blocks=3, texture_blocks=1, seed=0)
    model = snb.AutoRFMix(3, 1, D)
else:
    D = 128
    sd = oracle.init_codenerf_state(shape_blocks=5, texture_blocks=5, W=D, latent_dim=D, seed=0)
    model = snb.AutoRFMix()
model.load_state_dict(sd)
model = model.to(dev)
model.precision = a.precision
model.requires_grad_(False)
R = snb.renderer.NeRFRenderer(n_samples=64)
objs = bench.make_objects(100, a.objects, a.im_sz)
codes = [oracle.synthetic_latents(100 + i, 1, D) for i in range(a.objects)]
d = [dict(K=o["K"].to(dev), cam=o["cam_pose"].to(dev).requires_grad_(), wlh=o["wlh"], roi=o["roi"], tgt=o["img"].reshape(-1, 3).to(dev),
          occ=o["mask_occ"].reshape(-1, 1).to(dev), img=o["img"], mask=o["mask_occ"], shp=c[0].to(dev).requires_grad_(),
          tex=c[1].to(dev).requires_grad_())
     for o, c in zip(objs, codes)]
if a.path == "batched":
    cams = torch.stack([o["cam_pose"] for o in objs]).to(dev).requires_grad_()
    shps = torch.cat([c[0] for c in codes]).to(dev).requires_grad_()
    texs = torch.cat([c[1] for c in codes]).to(dev).requires_grad_()
    Ks = torch.stack([o["K"] for o in objs]).to(dev)
    ones = torch.ones(a.objects, device=dev)


def step():
    if a.path == "batched":
        cams.grad = shps.grad = texs.grad = None
        rgb, dep, acc, tgt, occ = R.render_rays_batch(model, dev, [o["img"] for o in objs], [o["mask_occ"] for o in objs], cams,
                                                      [o["wlh"] for o in objs], Ks, [o["roi"] for o in objs], shps, texs, im_sz=a.im_sz)
        snb.losses.refine_loss_batch(rgb, acc, tgt, occ, 0.1)[0].backward(gradient=ones)
        return
    for x in d:
        x["cam"].grad = x["shp"].grad = x["tex"].grad = None
        if a.path == "per-object":
            rgb, dep, acc, tgt, occ = R.render_rays(model, dev, x["img"], x["mask"], x["cam"], x["wlh"], x["K"], x["roi"], x["shp"], x["tex"],
                                                    im_sz=a.im_sz)
            snb.losses.refine_loss(rgb, acc, tgt, occ, 0.1)[0].backward()
            continue
        ro, vd = snb.utils.get_rays(x["K"], x["cam"], x["roi"], uv_steps=[a.im_sz, a.im_sz])
        xyz, vdr, zv, _ = R.prepare_sampled_rays(ro, vd, x["wlh"])
        sig, rgbs = model(xyz, vdr, x["shp"], x["tex"])
        rgb, dep, acc = R.volume_render(sig.squeeze(-1), rgbs, zv)
        bench.refine_loss(rgb, acc, x["tgt"], x["occ"]).backward()


for _ in range(a.warmup):
    step()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(a.steps):
    step()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / a.steps
rays = a.objects * a.im_sz ** 2
print("step_ms", ms, "objects", a.objects, "rays", rays, "rays_per_s", rays / ms * 1e3, "decoder", a.decoder, "path", a.path,
      "precision", a.precision, "SNB_FP32_SIMT", os.environ.get("SNB_FP32_SIMT", "0"))
