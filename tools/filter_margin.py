#!/usr/bin/env python
"""Margin of the closest-hit filter (csrc/pt_filter.cuh), measured on the GPU: for several scenes and ray
populations, compare the filtered closest hit with the exact scan at filter scales 1 ... 0 and print mismatches and
fallback rates.  The shipped scale is 1; the smallest scale with zero mismatches is the empirical safety factor.

usage: python tools/filter_margin.py [n_rays]"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
pt = importlib.import_module("project3-pathtracer_b200")
from scenes_for_tests import all_scenes, ray_sets  # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
    scales = [1.0, 0.5, 0.25, 0.125, 0.0625, 0.03125, 0.0]
    print("%-22s %-14s %s" % ("scene", "rays", "  ".join("s=%-7g" % s for s in scales)))
    for name, (g, m, cam) in all_scenes(pt).items():
        with pt.Context(g, m, cam) as ctx:
            for rname, (o, d) in ray_sets(pt, ctx, g, n).items():
                want = ctx.intersect(o, d, mode=pt.HIT_EXACT_SCAN)
                cells = []
                for s in scales:
                    ctx.set_filter_scale(s)
                    gid, t, p, nr, fb = ctx.intersect(o, d, with_stats=True)
                    hit = want[0] >= 0
                    bad = int((gid != want[0]).sum() + (t.view(np.uint32) != want[1].view(np.uint32)).sum()
                              + (p[hit].view(np.uint32) != want[2][hit].view(np.uint32)).any(axis=1).sum()
                              + (nr[hit].view(np.uint32) != want[3][hit].view(np.uint32)).any(axis=1).sum())
                    cells.append("%d/%.4f%%" % (bad, 100.0 * fb / len(gid)))
                ctx.set_filter_scale(1.0)
                print("%-22s %-14s %s" % (name, rname, "  ".join("%-9s" % c for c in cells)), flush=True)
            # primary rays through depth 0's closest hit (per-pixel table first, then the filter): the table's margin
            # scales with the filter's; cells = mismatches among all rays / share of rays the table decided
            if ctx.primary_table_info()[0]:
                spp = max(1, n // ctx.npix)
                pixel = np.tile(np.arange(ctx.npix, dtype=np.uint32), spp)
                sample = np.repeat(np.arange(spp, dtype=np.uint32), ctx.npix)
                o, d = ctx.raygen(565, pixel, sample)
                want = ctx.intersect(o, d, mode=pt.HIT_EXACT_SCAN)
                cells = []
                for s in scales:
                    ctx.set_filter_scale(s)
                    gid, t, p, nr, dec = ctx.primary_hit(565, pixel, sample)
                    hit = want[0] >= 0
                    bad = int(((gid != want[0]) | (t.view(np.uint32) != want[1].view(np.uint32))).sum()
                              + (p[hit].view(np.uint32) != want[2][hit].view(np.uint32)).any(axis=1).sum())
                    cells.append("%d/%.2f%%" % (bad, 100.0 * dec.mean()))
                ctx.set_filter_scale(1.0)
                print("%-22s %-14s %s" % (name, "primary", "  ".join("%-9s" % c for c in cells)), flush=True)


if __name__ == "__main__":
    main()
