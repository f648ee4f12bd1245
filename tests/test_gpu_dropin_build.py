"""The drop-in claim, executed: oracle/_ref/ref_dropin is a headless host compiled against the REFERENCE'S OWN
headers (src/scene.h, src/sceneStructs.h, src/raytraceKernel.h, src/image.h) and linked with the reference's own
scene.cpp / utilities.cpp / image.cpp -- and with libpt_b200.so in place of src/raytraceKernel.cu (oracle/Makefile
`dropin`, oracle/ref_dropin_main.cpp).  It runs the reference's per-iteration loop (src/main.cpp:93-139) and saves with
the reference's `image` class; the pixels must be the ones the C ABI produces for the same samples."""
import os
import subprocess

import numpy as np
import pytest
from PIL import Image

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "ref_dropin")


def test_reference_host_linked_against_libpt_b200(pt, sample_scene, tmp_path):
    if not os.path.exists(EXE):
        pytest.skip("oracle/_ref/ref_dropin not built (needs the reference checkout at build time: PT_REFERENCE_DIR, default /root/reference)")
    depth, seed, iters = 8, 565, 4
    out = tmp_path / "dropin.png"
    pbo = tmp_path / "pbo.raw"
    log = subprocess.check_output([EXE, "scene=" + os.path.join(ROOT, "scenes", "sample.txt"), "iterations=%d" % iters,
                                   "depth=%d" % depth, "seed=%d" % seed, "out=%s" % out, "pbo=%s" % pbo], text=True)
    assert "Saved frame 0" in log
    got = np.asarray(Image.open(tmp_path / "dropin.0.png").convert("RGB"))
    W, H = sample_scene["width"], sample_scene["height"]
    assert got.shape == (H, W, 3)
    # the same four samples through the C ABI, one per launch like the reference's loop (so every pixel's float sum
    # is formed in the same order and the comparison can be exact)
    with pt.Context(sample_scene["geoms"], sample_scene["materials"], sample_scene["camera"]) as ctx:
        ctx.set_wavefront_paths(W * H)
        for k in range(iters):
            ctx.render(k, 1, depth, seed)
        mean = ctx.download_mean(iters)
        rgba = ctx.resolve_rgba8(iters)
    want = pt.image_to_rgb8(mean, W, H)  # mirrored x + the reference writer's 8-bit rule (tests/test_image_writer.py)
    assert (got == want).all(), "pixels differ: %d of %d" % (int((got != want).any(axis=2).sum()), W * H)
    assert got.mean() > 5  # a real picture, not a black frame
    # the device buffer standing in for the mapped PBO holds sendImageToPBO's bytes of the running mean
    raw = np.fromfile(pbo, dtype=np.uint8).reshape(H * W, 4)
    assert (raw == np.asarray(rgba).reshape(H * W, 4)).all()
