#!/usr/bin/env python
"""The primary-ray table (csrc/pt_kernels.cuh: k_primary_table), measured on the GPU for the sample scene: the share
of primary rays its candidate settles, the share of depth-0 units (32 consecutive pixels of one sample) in which some
lane still runs the filter scan, the time of one table build at 800x800 and 3840x2160, and the mean time of the
depth-0 launch (k_bounce<true, false>) in a 64-spp render, from torch.profiler.

usage: python tools/primary_table_stats.py [--spp 16] [--kernel-only]
With --kernel-only only the depth-0 launch time is measured: that part also runs against builds without the table."""
import argparse
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
pt = importlib.import_module("project3-pathtracer_b200")
from conftest import with_resolution  # noqa: E402
from scenes_for_tests import _sample  # noqa: E402


def depth0_us(g, m, cam, spp=64, depth=8):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with pt.Context(g, m, cam) as ctx:
        ctx.render(0, spp, depth, 565)  # warm-up
        ctx.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.render(0, spp, depth, 565)
            ctx.sync()
    times = [e.device_time for e in prof.events() if "k_bounce<true, false" in e.name or "k_bounceILb1ELb0E" in e.name]
    return float(np.mean(times)), len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--kernel-only", action="store_true")
    args = ap.parse_args()
    g, m, cam = _sample(pt)
    out = {}
    us, n = depth0_us(g, m, cam)
    out["depth0_launch_us"] = us
    out["depth0_launches"] = n
    if not args.kernel_only:
        with pt.Context(g, m, cam) as ctx:
            W, H = ctx.width, ctx.height
            on, ms = ctx.primary_table_info(time_build=True)
            out["table_active"] = on
            out["build_ms_800"] = min(ms, ctx.primary_table_info(time_build=True)[1])
            pixel = np.tile(np.arange(ctx.npix, dtype=np.uint32), args.spp)
            sample = np.repeat(np.arange(args.spp, dtype=np.uint32), ctx.npix)
            _, _, _, _, dec, fb = ctx.primary_hit(565, pixel, sample, with_stats=True)
            out["decided"] = float(dec.mean())
            out["fallbacks"] = fb
            out["units_scanning"] = float((~dec.reshape(-1, 32)).any(axis=1).mean())
            out["pixels_without_candidate"] = float((~dec.reshape(args.spp, -1)).all(axis=0).mean())
        cam4k = with_resolution(cam, 3840, 2160)
        with pt.Context(g, m, cam4k) as ctx:
            ctx.primary_table_info(time_build=True)
            out["build_ms_4k"] = ctx.primary_table_info(time_build=True)[1]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
