"""GPU parity of glossy reflection (pt_set_glossy, pt_sample_glossy) against the C restatement: the lobe bit for bit,
renders through every bounce kernel that has a glossy variant (fused, re-batched, hierarchy; with and without direct
light sampling; with subsurface scattering), the furnace, the switch, the sample stream, the compat shim and the headless
driver.  Images are compared bit for bit where a pixel receives at most two contributions (float addition is
commutative), otherwise within 1e-5 of the pixel's sum (the GPU adds contributions with atomics in arbitrary order)."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLD, ROOT, f32, same_bits, with_resolution
from glossy_scenes import as_mirrors, furnace, glossy_hierarchy_scene, glossy_media_scene, glossy_scene

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering and glossy reflection (oracle/pt_oracle_glossy.c)"""
    from oracle_glossy import OracleGlossy
    return OracleGlossy()


def test_sample_glossy_matches_golden_vectors(pt):
    with open(os.path.join(GOLD, "glossy_vectors.json")) as f:
        gv = json.load(f)
    got = pt.sample_glossy(f32(gv["normal"]), f32(gv["incident"]), f32(gv["exponent"]), f32(gv["u"]))
    assert same_bits(got.ravel(), f32(gv["direction"]))


def test_sample_glossy_sweep_matches_oracle(pt, oracle):
    """every u0 = k 2^-24 the renderer can draw, with random normals, incident directions (grazing ones included),
    exponents and u1"""
    n = 1 << 24
    rng = np.random.default_rng(9)
    u = np.empty((n, 2), np.float32)
    u[:, 0] = (np.arange(n) * 2.0 ** -24).astype(np.float32)
    u[:, 1] = (rng.integers(0, 1 << 24, n) * 2.0 ** -24).astype(np.float32)
    nrm = rng.normal(size=(n, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    e = np.exp(rng.uniform(np.log(1e-3), np.log(1e5), n)).astype(np.float32)
    got = pt.sample_glossy(nrm, d, e, u)
    want = oracle.sample_glossy(nrm, d, e, u)
    assert same_bits(got, want)


def _render(pt, oracle, g, m, cam, spp, depth, seed, policy=0, nee=False, sss=False, first=0):
    want, want_live, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss, glossy=True),
                                       first, spp, depth, seed)
    with pt.Context(g, m, cam) as c:
        c.set_kernel_policy(policy)
        c.set_direct_lighting(nee)
        c.set_subsurface(sss)
        c.set_glossy(True)
        c.render(first, spp, depth, seed)
        got = c.download_sum()
        _, _, live = c.counters()
    assert live[:depth].tolist() == want_live.tolist()
    return got, want


@pytest.mark.parametrize("policy", [1, 2])
def test_glossy_render_bit_identical(pt, oracle, sample_scene, policy):
    """few geoms: k_bounce at depth 0 (the primary-ray table stays on), then the re-batched k_bounce_q (policy 1) or the
    fused k_bounce (policy 2)"""
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 96, 96)
    got, want = _render(pt, oracle, g, m, cam, 2, 10, 17, policy=policy)
    assert same_bits(got, want)
    mirror, _, _ = oracle.render(oracle.make_scene(g, as_mirrors(m), cam), 0, 2, 10, 17)
    assert not same_bits(got, mirror)  # (the lobes changed the image)


def test_glossy_keeps_the_primary_table(pt, sample_scene):
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 64)
    with pt.Context(g, m, cam) as c:
        c.set_glossy(True)
        assert c.primary_table_info()[0]
        c.render(0, 1, 4, 2)
        assert c.primary_table_info()[0]


def test_glossy_hierarchy_render_bit_identical(pt, oracle, sample_scene):
    g, m = glossy_hierarchy_scene(pt, sample_scene)
    assert len(g) >= 33
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want = _render(pt, oracle, g, m, cam, 2, 10, 3)
    assert same_bits(got, want)


@pytest.mark.parametrize("scene", ["few", "hierarchy"])
def test_glossy_with_direct_lighting(pt, oracle, sample_scene, scene):
    """direct light sampling and glossy reflection together: two-segment paths bit for bit (at most two contributions per
    pixel), deeper ones within 1e-5"""
    g, m = glossy_scene(pt, sample_scene) if scene == "few" else glossy_hierarchy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want = _render(pt, oracle, g, m, cam, 1, 2, 9, nee=True)
    assert same_bits(got, want)
    for policy in (1, 2):
        got, want = _render(pt, oracle, g, m, cam, 2, 8, 9, policy=policy, nee=True)
        assert np.allclose(got, want, rtol=SUM_TOL, atol=SUM_TOL)


@pytest.mark.parametrize("policy", [1, 2])
def test_glossy_with_subsurface(pt, oracle, sample_scene, policy):
    """glossy reflectors and scattering media in one scene: the variants with both switches"""
    g, m = glossy_media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want = _render(pt, oracle, g, m, cam, 2, 10, 21, policy=policy, sss=True)
    assert same_bits(got, want)
    got, want = _render(pt, oracle, g, m, cam, 1, 2, 21, policy=policy, sss=True, nee=True)
    assert same_bits(got, want)


def test_furnace(pt, oracle, sample_scene):
    """a glossy sphere of SPECRGB 0.5 in an emissive box: pixel sums of exactly spp (walls) or spp / 2 (the sphere), the
    oracle's image"""
    w = h = 48
    spp = 4
    g, m, cam = furnace(pt, sample_scene["camera"], w, h)
    with pt.Context(g, m, cam) as c:
        c.set_glossy(True)
        c.render(0, spp, 8, 3)
        img = c.download_sum()
        _, _, live = c.counters()
    k = 2 * (spp - img[:, 0])
    assert (k == np.round(k)).all() and (k >= 0).all() and (k <= spp).all()
    assert (img[:, 0] == spp).sum() > 0 and (img[:, 0] == spp / 2).sum() > 0.2 * w * h
    want, want_live, _ = oracle.render(oracle.make_scene(g, m, cam, glossy=True), 0, spp, 8, 3)
    assert same_bits(img, want) and live[:8].tolist() == want_live.tolist()


def test_switch(pt, sample_scene):
    """off with SPECEX > 0 = SPECEX 0 (off or on) -- the mirror; on with SPECEX > 0 differs"""
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 64)
    out = []
    for mats, on in ((m, False), (as_mirrors(m), False), (as_mirrors(m), True), (m, True)):
        with pt.Context(g, mats, cam) as c:
            c.set_glossy(on)
            c.render(0, 2, 8, 4)
            out.append((c.download_sum(), c.counters()[2]))
    for img, live in out[1:3]:
        assert same_bits(img, out[0][0]) and (live == out[0][1]).all()
    assert not same_bits(out[3][0], out[0][0])


@pytest.mark.parametrize("group", [1, 3])
def test_sample_stream_with_glossy(pt, sample_scene, group):
    """pt_stream_* with the switch on leaves exactly the sums of one pt_render per sample"""
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 48)
    depth, seed, n = 8, 12, 9
    with pt.Context(g, m, cam) as a, pt.Context(g, m, cam) as b:
        for c in (a, b):
            c.set_glossy(True)
        b.stream_begin(0, 0, depth, seed, group)
        for k in range(n):
            a.render(k, 1, depth, seed)
            mean, spp = b.stream_next()
            assert spp == k + 1 and same_bits(mean, a.download_mean(k + 1)), k
        b.stream_end()
        assert same_bits(b.download_sum(), a.download_sum())


def test_cudaRaytraceCore_glossy_switch_restarts_the_stream(pt, oracle, sample_scene):
    """compat.set_glossy changes the estimator for the calls that follow: samples traced ahead with the old setting are
    dropped"""
    compat = importlib.import_module("project3-pathtracer_b200.compat")
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 64)
    rs = compat.RefScene([(g, cam)], m, iterations=4)
    compat.reset(); compat.set_trace_depth(8); compat.set_seed(6); compat.set_exit_on_error(False)
    call = lambda k: compat.cudaRaytraceCore(None, rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))  # noqa: E731
    on, off = oracle.make_scene(g, m, cam, glossy=True), oracle.make_scene(g, m, cam)
    want = np.zeros((64 * 64, 3), np.float32)
    try:
        compat.set_glossy(True)
        for k in (1, 2):
            call(k)
            oracle.render(on, k - 1, 1, 8, 6, sum_rgb=want)
        assert same_bits(rs.image, want / np.float32(2))
        compat.set_glossy(False)  # sample 2 was traced ahead with glossy lobes: it must not count
        call(3)
        oracle.render(off, 2, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(3), rtol=1e-6, atol=1e-6)
        compat.set_glossy(True)
        call(4)
        oracle.render(on, 3, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(4), rtol=1e-6, atol=1e-6)
        assert compat.last_status() == 0
    finally:
        compat.set_glossy(False)
        compat.reset()


def test_headless_driver_glossy_switch(pt, tmp_path):
    """pt_render scene=scenes/cornell_glossy.txt glossy=1 (reduced): the segments and image the C ABI renders"""
    sys.path.insert(0, os.path.join(ROOT, "scenes"))
    import gen_scenes
    from PIL import Image
    p = tmp_path / "glossy.txt"
    p.write_text(gen_scenes.cornell_glossy().replace("RES         800 800", "RES         96 64"))
    g, m, cam, lens = pt.Scene(p).frame(0)
    exe = os.path.join(ROOT, "project3-pathtracer_b200", "pt_render")
    imgs = []
    for on in (1, 0):
        out = subprocess.check_output([exe, "scene=%s" % p, "spp=2", "depth=8", "seed=8", "glossy=%d" % on,
                                       "out=%s" % (tmp_path / ("g%d.png" % on)), "json=1"], text=True)
        info = json.loads(out.strip().splitlines()[-1])
        with pt.Context(g, m, cam, lens) as c:
            c.set_glossy(bool(on))
            c.render(0, 2, 8, 8)
            want_sum = c.download_sum()
            _, segs, _ = c.counters()
        assert info["segments"] == int(segs)
        got8 = np.asarray(Image.open(info["file"]).convert("RGB"))
        assert (got8 == pt.image_to_rgb8(want_sum / np.float32(2), 96, 64)).all()
        imgs.append(got8)
    assert (imgs[0] != imgs[1]).any()
