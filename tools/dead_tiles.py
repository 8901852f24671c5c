#!/usr/bin/env python
"""Share of the batched render's decoder-backward work whose upstream gradient is exactly zero, for bench.py's workload (CPU only).

The refine loss weights every ray by |occ|, so a ray with occ == 0 feeds its decoder rows a zero gradient; pad rows get none
either.  The batched render (csrc/render_batch.cu) lays out each object's rows as: the hit rays in pixel order with S rows each,
then one row per miss ray, padded to 256 rows.  This script rebuilds that layout from the oracle's slab test and counts the rows,
128-row tiles and 256-row super tiles (the unit the decoder backward skips) in which every row is dead.

  python tools/dead_tiles.py [--objects 16] [--im 128] [--samples 64] [--seed0 100]
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle  # noqa: E402
from supnerf_b200 import synthetic  # noqa: E402  (bench.py's seeded objects)


def object_rows(obj, im, S):
    """Per decoder row of one object (padded to 256): True where the row's upstream gradient can be nonzero."""
    ro, vd = oracle.get_rays(obj["K"], obj["cam_pose"], obj["roi"], uv_steps=[im, im])
    diag, half = oracle.box_constants(obj["wlh"])
    hb = torch.from_numpy(half)
    hit = oracle.ray_box_intersection(ro / (diag / 2), vd, -hb.expand_as(ro), hb.expand_as(ro))[2].numpy().astype(bool)
    occ = obj["mask_occ"].reshape(-1).numpy()
    live_ray = occ != 0
    rows = np.concatenate([np.repeat(live_ray[hit], S), live_ray[~hit]])
    pad = -len(rows) % 256
    return np.concatenate([rows, np.zeros(pad, dtype=bool)])


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--objects", type=int, default=16)
    ap.add_argument("--im", type=int, default=128)
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--seed0", type=int, default=100)
    a = ap.parse_args()
    live = np.concatenate([object_rows(synthetic.synthetic_object(a.seed0 + i, im_sz=a.im), a.im, a.samples) for i in range(a.objects)])
    print("rows executed per launch: %d" % len(live))
    for name, g in (("rows", 1), ("128-row tiles", 128), ("256-row super tiles", 256)):
        units = live.reshape(-1, g).any(axis=1)
        dead = int((~units).sum())
        print("%-20s dead %9d of %9d  (%.1f %%)" % (name, dead, len(units), 100.0 * dead / len(units)))


if __name__ == "__main__":
    main()
