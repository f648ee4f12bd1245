#!/usr/bin/env python
"""Russian roulette's cost and benefit: for each workload, roulette off and from depth k in {1, 3}, at max_depth 8 and 32.
Workloads: scenes/sample.txt, scenes/cornell_glass_dof.txt and scenes/cornell_sss.txt with subsurface scattering on.
Device-event timing (pt_last_render_ms) of `reps` renders of `spp` samples each after one warm-up render; per setting it
reports milliseconds, segments, Gseg/s and spp/s, the relative MSE against a reference image rendered in the same run
(roulette off, 16x the spp, a sample range disjoint from the measured one), and efficiency = 1 / (MSE x ms).  Prints one
JSON line, with the card's name and power limit read in the same run.

Usage: python tools/bench_roulette.py [--spp 16] [--reps 3] [--scale 4]"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pt = importlib.import_module("project3-pathtracer_b200")

WORKLOADS = [("scenes/sample.txt", False), ("scenes/cornell_glass_dof.txt", False), ("scenes/cornell_sss.txt", True)]


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=int, default=4, help="divide each scene's resolution by this (the reference costs 16x)")
    a = ap.parse_args()
    if pt.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    res = {"spp": a.spp, "reps": a.reps, "scale": a.scale, "workloads": []}
    ref_first = 1 << 20  # the reference's samples: disjoint from the measured ones
    for path, sss in WORKLOADS:
        scene = pt.Scene(os.path.join(ROOT, path))
        g, m, cam, lens = scene.frame(0)
        cam = cam.copy()
        w, h = scene.width // a.scale, scene.height // a.scale
        cam["resolution"][0] = [w, h]
        for depth in (8, 32):
            row = {"scene": path, "subsurface": sss, "width": w, "height": h, "depth": depth}
            with pt.Context(g, m, cam, lens) as c:
                c.set_subsurface(sss)
                c.set_russian_roulette(0)
                c.clear()
                c.render(ref_first, 16 * a.spp * a.reps, depth, 1)
                ref = c.download_sum().astype(np.float64) / (16 * a.spp * a.reps)
                for k in (0, 1, 3):
                    c.set_russian_roulette(k)
                    c.clear()
                    c.render(0, a.spp, depth, 1)  # warm-up: module load, first-wavefront policy
                    c.sync()
                    c.clear()
                    ms = []
                    for r in range(a.reps):
                        c.render(r * a.spp, a.spp, depth, 1)
                        ms.append(c.last_render_ms())
                    img = c.download_sum().astype(np.float64) / (a.spp * a.reps)
                    _, segs, _ = c.counters()
                    total = sum(ms)
                    mse = float(np.mean((img - ref) ** 2) / max(np.mean(ref ** 2), 1e-30))
                    row["rr%d" % k] = {"ms_per_render": [round(x, 3) for x in ms], "segments": int(segs),
                                       "gseg_per_s": round(segs / total / 1e6, 3),
                                       "spp_per_s": round(a.spp * a.reps / (total / 1e3), 2), "rel_mse": mse,
                                       "efficiency": 1.0 / (mse * total / a.reps) if mse > 0 else None}
            res["workloads"].append(row)
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
