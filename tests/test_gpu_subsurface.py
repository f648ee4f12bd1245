"""GPU parity of subsurface scattering (pt_set_subsurface, pt_sample_medium) against the C restatement: the free flight
bit for bit, renders through every bounce kernel that has a medium variant (fused, re-batched, hierarchy; with and
without direct light sampling), the white furnace, the switch, the sample stream and the headless driver.
Images are compared bit for bit where a pixel receives at most two contributions (float addition is commutative),
otherwise within 1e-5 of the pixel's sum (the GPU adds contributions with atomics in arbitrary order)."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLD, ROOT, f32, same_bits, with_resolution
from medium_scenes import furnace, media_hierarchy_scene, media_scene

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering (oracle/pt_oracle_medium.c)"""
    from oracle_medium import OracleMedium
    return OracleMedium()


def test_sample_medium_matches_golden_vectors(pt):
    with open(os.path.join(GOLD, "medium_vectors.json")) as f:
        gv = json.load(f)
    flag, s, dirs, w = pt.sample_medium(f32(gv["absorption"]), f32(gv["scatter"]), f32(gv["distance"]), f32(gv["u"]))
    assert flag.astype(int).tolist() == gv["scattered"]
    for got, key in ((s, "s"), (dirs, "direction"), (w, "weight")):
        assert same_bits(got.ravel(), f32(gv[key])), key


def test_sample_medium_free_flight_sweep_matches_oracle(pt, oracle):
    """every xf = k 2^-24 the renderer can draw, with random directions' uniforms, absorption and segment lengths"""
    n = 1 << 24
    rng = np.random.default_rng(8)
    u = np.empty((n, 3), np.float32)
    u[:, :2] = (rng.integers(0, 1 << 24, (n, 2)) * 2.0 ** -24).astype(np.float32)
    u[:, 2] = (np.arange(n) * 2.0 ** -24).astype(np.float32)
    ab = rng.uniform(0, 4, (n, 3)).astype(np.float32)
    sc = np.full(n, 2.5, np.float32)
    d = rng.uniform(0.01, 8, n).astype(np.float32)
    got = pt.sample_medium(ab, sc, d, u)
    want = oracle.sample_medium(ab, sc, d, u)
    assert (got[0] == want[0]).all() and 0 < got[0].mean() < 1
    for g, w_ in zip(got[1:], want[1:]):
        assert same_bits(g, w_)


def _render(pt, oracle, g, m, cam, spp, depth, seed, policy=0, nee=False, first=0):
    want, want_live, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=True), first, spp, depth, seed)
    with pt.Context(g, m, cam) as c:
        c.set_kernel_policy(policy)
        c.set_direct_lighting(nee)
        c.set_subsurface(True)
        c.render(first, spp, depth, seed)
        got = c.download_sum()
        _, _, live = c.counters()
    assert live[:depth].tolist() == want_live.tolist()
    return got, want


@pytest.mark.parametrize("policy", [1, 2])
def test_media_render_bit_identical(pt, oracle, sample_scene, policy):
    """few geoms: k_bounce at depth 0, then the re-batched k_bounce_q (policy 1) or the fused k_bounce (policy 2)"""
    g, m = media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 96, 96)
    got, want = _render(pt, oracle, g, m, cam, 2, 10, 17, policy=policy)
    assert same_bits(got, want)
    plain, _, _ = oracle.render(oracle.make_scene(g, m, cam), 0, 2, 10, 17)
    assert not same_bits(got, plain)  # (the media changed the image)


def test_media_hierarchy_render_bit_identical(pt, oracle, sample_scene):
    g, m = media_hierarchy_scene(pt, sample_scene)
    assert len(g) >= 33
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want = _render(pt, oracle, g, m, cam, 2, 10, 3)
    assert same_bits(got, want)


@pytest.mark.parametrize("scene", ["few", "hierarchy"])
def test_media_with_direct_lighting(pt, oracle, sample_scene, scene):
    """direct light sampling and subsurface scattering together: two-segment paths bit for bit (at most two contributions
    per pixel), deeper ones within 1e-5"""
    g, m = media_scene(pt, sample_scene) if scene == "few" else media_hierarchy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want = _render(pt, oracle, g, m, cam, 1, 2, 9, nee=True)
    assert same_bits(got, want)
    for policy in (1, 2):
        got, want = _render(pt, oracle, g, m, cam, 2, 8, 9, policy=policy, nee=True)
        assert np.allclose(got, want, rtol=SUM_TOL, atol=SUM_TOL)


def test_white_furnace(pt, oracle, sample_scene):
    w = h = 48
    spp, depth = 2, 64
    g, m, cam = furnace(pt, sample_scene["camera"], w, h)
    with pt.Context(g, m, cam) as c:
        c.set_subsurface(True)
        c.render(0, spp, depth, 7)
        img = c.download_sum()
        _, segs, live = c.counters()
        c.set_subsurface(False)
        c.clear()
        c.render(0, spp, depth, 7)
        _, segs_glass, _ = c.counters()
    assert (img == np.round(img)).all() and (img[:, 0] == img[:, 1]).all()
    assert img[:, 0].sum() >= (1 - 1e-4) * w * h * spp
    assert segs > 1.5 * segs_glass
    want, want_live, _ = oracle.render(oracle.make_scene(g, m, cam, subsurface=True), 0, spp, depth, 7)
    assert same_bits(img, want) and live[:depth].tolist() == want_live.tolist()


def test_switch_off_equals_scatter_free_materials(pt, sample_scene):
    g, m = media_scene(pt, sample_scene)
    m0 = m.copy()
    m0["hasScatter"] = 0
    cam = with_resolution(sample_scene["camera"], 64, 64)
    out = []
    for mats, sss in ((m, False), (m0, False), (m0, True), (m, True)):
        with pt.Context(g, mats, cam) as c:
            c.set_subsurface(sss)
            c.render(0, 2, 8, 4)
            out.append((c.download_sum(), c.counters()[2]))
    for img, live in out[1:3]:
        assert same_bits(img, out[0][0]) and (live == out[0][1]).all()
    assert not same_bits(out[3][0], out[0][0])


@pytest.mark.parametrize("group", [1, 3])
def test_sample_stream_with_subsurface(pt, sample_scene, group):
    """pt_stream_* with the switch on leaves exactly the sums of one pt_render per sample"""
    g, m = media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 48)
    depth, seed, n = 8, 12, 9
    with pt.Context(g, m, cam) as a, pt.Context(g, m, cam) as b:
        for c in (a, b):
            c.set_subsurface(True)
        b.stream_begin(0, 0, depth, seed, group)
        for k in range(n):
            a.render(k, 1, depth, seed)
            mean, spp = b.stream_next()
            assert spp == k + 1 and same_bits(mean, a.download_mean(k + 1)), k
        b.stream_end()
        assert same_bits(b.download_sum(), a.download_sum())


def test_cudaRaytraceCore_subsurface_switch_restarts_the_stream(pt, oracle, sample_scene):
    """compat.set_subsurface changes the estimator for the calls that follow: samples traced ahead with the old setting
    are dropped"""
    compat = importlib.import_module("project3-pathtracer_b200.compat")
    g, m = media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 64)
    rs = compat.RefScene([(g, cam)], m, iterations=4)
    compat.reset(); compat.set_trace_depth(8); compat.set_seed(6); compat.set_exit_on_error(False)
    call = lambda k: compat.cudaRaytraceCore(None, rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))  # noqa: E731
    on, off = oracle.make_scene(g, m, cam, subsurface=True), oracle.make_scene(g, m, cam)
    want = np.zeros((64 * 64, 3), np.float32)
    try:
        compat.set_subsurface(True)
        for k in (1, 2):
            call(k)
            oracle.render(on, k - 1, 1, 8, 6, sum_rgb=want)
        assert same_bits(rs.image, want / np.float32(2))
        compat.set_subsurface(False)  # sample 2 was traced ahead with media: it must not count
        call(3)
        oracle.render(off, 2, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(3), rtol=1e-6, atol=1e-6)
        compat.set_subsurface(True)
        call(4)
        oracle.render(on, 3, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(4), rtol=1e-6, atol=1e-6)
        assert compat.last_status() == 0
    finally:
        compat.set_subsurface(False)
        compat.reset()


def test_headless_driver_sss_switch(pt, oracle, tmp_path):
    """pt_render scene=scenes/cornell_sss.txt sss=1 (reduced): the oracle's segments and image"""
    sys.path.insert(0, os.path.join(ROOT, "scenes"))
    import gen_scenes
    p = tmp_path / "sss.txt"
    p.write_text(gen_scenes.cornell_sss().replace("RES         800 800", "RES         96 64"))
    g, m, cam, lens = pt.Scene(p).frame(0)
    exe = os.path.join(ROOT, "project3-pathtracer_b200", "pt_render")
    imgs = []
    for sss in (1, 0):
        out = subprocess.check_output([exe, "scene=%s" % p, "spp=2", "depth=8", "seed=8", "sss=%d" % sss,
                                       "out=%s" % (tmp_path / ("s%d.png" % sss)), "json=1"], text=True)
        info = json.loads(out.strip().splitlines()[-1])
        want_sum, live, _ = oracle.render(oracle.make_scene(g, m, cam, lens, subsurface=bool(sss)), 0, 2, 8, 8)
        assert info["segments"] == int(live.sum())
        from PIL import Image
        got8 = np.asarray(Image.open(info["file"]).convert("RGB"))
        assert (got8 == pt.image_to_rgb8(want_sum / np.float32(2), 96, 64)).all()
        imgs.append(got8)
    assert (imgs[0] != imgs[1]).any()
