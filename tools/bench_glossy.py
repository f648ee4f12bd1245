#!/usr/bin/env python
"""Glossy reflection's cost: scenes/cornell_glossy.txt (800x800, three glossy spheres, a glossy wall and a mirror sphere in a
closed room) rendered with pt_set_glossy on and off (off: the same geoms as perfect mirrors).  Device-event timing
(pt_last_render_ms) of `reps` renders of `spp` samples each after one warm-up render; prints one JSON line with Gseg/s,
milliseconds and segments per setting, and the card's name and power limit read in the same run.

Usage: python tools/bench_glossy.py [--spp 64] [--depth 8] [--reps 3]"""
import argparse
import importlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pt = importlib.import_module("project3-pathtracer_b200")


def card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power = (x.strip() for x in out.split(","))
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--depth", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if pt.device_count() < 1:
        raise SystemExit("no CUDA device: nothing to measure")
    scene = pt.Scene(os.path.join(ROOT, "scenes", "cornell_glossy.txt"))
    g, m, cam, lens = scene.frame(0)
    res = {"scene": "scenes/cornell_glossy.txt", "width": scene.width, "height": scene.height, "spp": a.spp,
           "depth": a.depth, "reps": a.reps}
    with pt.Context(g, m, cam, lens) as c:
        for on in (True, False):
            c.set_glossy(on)
            c.clear()
            c.render(0, a.spp, a.depth, 1)  # warm-up: module load, first-wavefront policy
            c.sync()
            ms = []
            c.clear()
            for r in range(a.reps):
                c.render((r + 1) * a.spp, a.spp, a.depth, 1)
                ms.append(c.last_render_ms())
            _, segs, _ = c.counters()
            total = sum(ms)
            res["on" if on else "off"] = {"ms_per_render": [round(x, 3) for x in ms], "segments": int(segs),
                                          "segments_per_render": int(segs) // a.reps,
                                          "gseg_per_s": round(segs / total / 1e6, 3)}
    res["gpu"], res["power_limit"] = card()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
