#!/usr/bin/env python
"""Times the decoder C-ABI calls alone (CUDA events, current stream): fwd and bwd at 1 object x 16384 rays x 64 samples.
  python tools/time_decoder.py [precision] [--blocks S T] [--W W] [--latent-dim D]
Default: the bench decoder, 3 + 1 blocks at W = latent_dim = 256.  AutoRFMix() class defaults: --blocks 5 5 --W 128 --latent-dim 128.
SNB_FP32_SIMT=1 in the environment runs fp32 mode on the FFMA back end (no kernel-only line: it records no kernel events)."""
import argparse, os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import supnerf_b200 as snb
from oracle import oracle
ap = argparse.ArgumentParser()
ap.add_argument("precision", nargs="?", default="bf16")
ap.add_argument("--blocks", type=int, nargs=2, default=[3, 1], metavar=("SHAPE", "TEXTURE"))
ap.add_argument("--W", type=int, default=256)
ap.add_argument("--latent-dim", type=int, default=256)
a = ap.parse_args()
Bs, Bt, W, D = a.blocks[0], a.blocks[1], a.W, a.latent_dim
dev = "cuda"
sd = oracle.init_codenerf_state(shape_blocks=Bs, texture_blocks=Bt, W=W, latent_dim=D, seed=0)
m = snb.AutoRFMix(Bs, Bt, W) if W == D else snb.CodeNeRF(Bs, Bt, W=W, latent_dim=D)
m.load_state_dict(sd); m = m.to(dev); m.precision = a.precision; m.requires_grad_(False)
# algorithmic multiply-adds per sample (BASELINE.md): encoding_xyz, shape layers, encoding_shape, sigma, encoding_viewdir, texture
# layers, rgb.0, rgb head; the per-object latent layers are not per sample.  3 + 1 at W = 256: 449 664
dx, dv = 63, 27
MAC = dx * W + Bs * W * W + W * W + W + (W + dv) * W + Bt * W * W + W * (W // 2) + (W // 2) * 3
N, S = 16384, 64
g = torch.Generator().manual_seed(0)
xyz = ((torch.rand(N, S, 3, generator=g) - 0.5) * 1.6).to(dev).requires_grad_()
vd = torch.nn.functional.normalize(torch.randn(N, 1, 3, generator=g), dim=-1).repeat(1, S, 1).to(dev).requires_grad_()
shp, tex = [t.to(dev).requires_grad_() for t in oracle.synthetic_latents(0, 1, D)]
def run(n):
    tf, tb = [], []
    for _ in range(n):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record(); sig, rgb = m(xyz, vd, shp, tex); e[1].record()
        gs, gr = torch.ones_like(sig), torch.ones_like(rgb)
        e[2].record(); torch.autograd.grad([sig, rgb], [xyz, vd, shp, tex], [gs, gr]); e[3].record()
        torch.cuda.synchronize()
        tf.append(e[0].elapsed_time(e[1])); tb.append(e[2].elapsed_time(e[3]))
    return min(tf), min(tb)
run(3)
import ctypes
lib = snb._lib.load()
hnd = m._handle(xyz.device).h
lib.snb_kernel_timing_enable(hnd, 1)
f, b = run(10)
buf = (ctypes.c_float * 64)()
kf = [buf[i] for i in range(lib.snb_kernel_timing_read(hnd, 0, buf, 64))]
kb = [buf[i] for i in range(lib.snb_kernel_timing_read(hnd, 1, buf, 64))]
lib.snb_kernel_timing_enable(hnd, 0)
fl = 2 * MAC * N * S / 1e12
print(f"decoder {Bs}+{Bt} blocks, W = {W}, latent_dim = {D}, {MAC} MAC / sample, precision {a.precision}, SNB_FP32_SIMT={os.environ.get('SNB_FP32_SIMT', '0')}")
if kf: print(f"   kernel only: fwd {min(kf):.3f} ms ({fl/min(kf)*1e3:.0f} TF/s)  bwd {min(kb):.3f} ms ({fl/min(kb)*1e3:.0f} TF/s)")
print(f"SNB_TC_EXP={os.environ.get('SNB_TC_EXP','0')} fwd {f:.3f} ms ({fl/f*1e3:.0f} TF/s)  bwd {b:.3f} ms ({fl/b*1e3:.0f} TF/s)")
