"""bench.py end to end at a small sample count: --steps sets the number of timed steps (their launches are counted) and
--dump-outputs writes the arrays one step computes.  A step clears the image before it renders, so every step computes
the same arrays, and the dump must equal one direct render through the C ABI (not the sum of several steps)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import same_bits

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_equal_a_direct_render(pt, sample_scene, tmp_path):
    spp, depth, seed, steps = 2, 8, 565, 2
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "0",
                                   "--spp", str(spp), "--wf-spp", str(spp), "--no-extras", "--no-cpu-baseline",
                                   "--dump-outputs", str(tmp_path)], cwd=ROOT, text=True)
    line = json.loads(out.strip().splitlines()[-1])
    img = np.load(tmp_path / "image_sum.npy")
    live = np.load(tmp_path / "live_per_depth.npy")
    assert img.dtype == np.float32 and live.dtype == np.float64
    with pt.Context(sample_scene["geoms"], sample_scene["materials"], sample_scene["camera"]) as c:
        c.set_wavefront_paths(c.npix * spp)
        l0 = c.launch_count()
        c.clear()
        c.render(0, spp, depth, seed)
        launches = c.launch_count() - l0
        want = c.download_sum()
        _, _, want_live = c.counters()
    assert line["steps"] == steps and line["gpu_launches"] == steps * launches
    assert live.tolist() == want_live[:depth].astype(np.float64).tolist()
    assert same_bits(img, want)  # at most two contributions per pixel: the sum does not depend on their order
