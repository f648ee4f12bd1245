"""GPU parity of Russian roulette (pt_set_russian_roulette) against the C restatement: renders through every bounce kernel
that has a roulette variant (re-batched, fused, hierarchy; with direct light sampling; with subsurface scattering and
glossy reflection), the switch, unbiasedness, the sample stream, the compat shim and the headless driver.  Images are
compared bit for bit where a pixel receives at most two contributions (float addition is commutative), otherwise within
1e-5 of the pixel's sum (the GPU adds contributions with atomics in arbitrary order)."""
import importlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, same_bits, with_resolution
from glossy_scenes import glossy_hierarchy_scene, glossy_media_scene, glossy_scene
from roulette_scenes import batch_means, closed_room, white, within_standard_errors

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering, glossy reflection and Russian roulette
    (oracle/pt_oracle_roulette.c)"""
    from oracle_roulette import OracleRoulette
    return OracleRoulette()


def _render(pt, oracle, g, m, cam, spp, depth, seed, k, policy=0, nee=False, sss=False, glossy=False):
    want, want_live, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss, glossy=glossy,
                                                         roulette=k), 0, spp, depth, seed)
    with pt.Context(g, m, cam) as c:
        c.set_kernel_policy(policy)
        c.set_direct_lighting(nee)
        c.set_subsurface(sss)
        c.set_glossy(glossy)
        c.set_russian_roulette(k)
        c.render(0, spp, depth, seed)
        got = c.download_sum()
        _, _, live = c.counters()
    assert live[:depth].tolist() == want_live.tolist()
    return got, want, want_live


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("policy", [1, 2])
def test_roulette_render_bit_identical(pt, oracle, sample_scene, policy, k):
    """few geoms: the re-batched k_bounce_q (policy 1) or the fused k_bounce (policy 2) from depth k on"""
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = with_resolution(sample_scene["camera"], 96, 96)
    got, want, live = _render(pt, oracle, g, m, cam, 2, 12, 17, k, policy=policy)
    assert same_bits(got, want)
    _, off, _ = oracle.render(oracle.make_scene(g, m, cam), 0, 2, 12, 17)
    assert live.sum() < off.sum()  # (the roulette ended paths)


def test_roulette_hierarchy_render_bit_identical(pt, oracle, sample_scene):
    g, m = glossy_hierarchy_scene(pt, sample_scene)
    assert len(g) >= 33
    cam = with_resolution(sample_scene["camera"], 80, 80)
    for k in (1, 2):
        got, want, _ = _render(pt, oracle, g, m, cam, 2, 10, 3, k)
        assert same_bits(got, want)
    got, want, _ = _render(pt, oracle, g, m, cam, 2, 10, 3, 1, glossy=True)
    assert same_bits(got, want)


@pytest.mark.parametrize("scene", ["few", "hierarchy"])
def test_roulette_with_direct_lighting(pt, oracle, sample_scene, scene):
    """live[] exact, images within 1e-5 of the pixel sum"""
    g, m = glossy_scene(pt, sample_scene) if scene == "few" else glossy_hierarchy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 80, 80)
    for policy in (1, 2):
        got, want, _ = _render(pt, oracle, g, m, cam, 2, 8, 9, 1, policy=policy, nee=True)
        assert np.allclose(got, want, rtol=SUM_TOL, atol=SUM_TOL)


@pytest.mark.parametrize("policy", [1, 2])
def test_roulette_with_subsurface_and_glossy(pt, oracle, sample_scene, policy):
    """media and glossy reflectors in one scene: the variants with every switch"""
    g, m = glossy_media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 80, 80)
    got, want, _ = _render(pt, oracle, g, m, cam, 2, 10, 21, 1, policy=policy, sss=True, glossy=True)
    assert same_bits(got, want)
    got, want, _ = _render(pt, oracle, g, m, cam, 2, 10, 21, 2, policy=policy, sss=True, glossy=True, nee=True)
    assert np.allclose(got, want, rtol=SUM_TOL, atol=SUM_TOL)


def test_switch(pt, sample_scene):
    """off = k 0 = k >= max_depth - 1 = a white scene with roulette on; on differs on the sample scene; -1 and 64 are
    rejected"""
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = with_resolution(sample_scene["camera"], 64, 64)
    depth = 8

    def run(mats, k):
        with pt.Context(g, mats, cam) as c:
            if k is not None:
                c.set_russian_roulette(k)
            c.render(0, 2, depth, 4)
            return c.download_sum(), c.counters()[2]

    off = run(m, None)
    for k in (0, depth - 1, 63):
        img, live = run(m, k)
        assert same_bits(img, off[0]) and (live == off[1]).all(), k
    w_off = run(white(m), None)
    w_on = run(white(m), 1)
    assert same_bits(w_on[0], w_off[0]) and (w_on[1] == w_off[1]).all()
    on = run(m, 1)
    assert not same_bits(on[0], off[0]) and on[1].sum() < off[1].sum()
    with pt.Context(g, m, cam) as c:
        for bad in (-1, 64):
            with pytest.raises(pt.PtError):
                c.set_russian_roulette(bad)


def test_unbiased(pt, sample_scene):
    """a closed diffuse room with a light at depth 16: batch means with roulette from depth 1 agree with roulette off
    within 4 combined standard errors"""
    g, m, cam = closed_room(pt, sample_scene["camera"], 64, 64)

    def run(k):
        with pt.Context(g, m, cam) as c:
            c.set_russian_roulette(k)

            def render(first, spp):
                c.clear()
                c.render(first, spp, 16, 77)
                return c.download_sum()

            return batch_means(render, 32, 16)

    off, on = run(0), run(1)
    ok, a, b, se = within_standard_errors(on, off)
    assert ok, (a, b, se)


@pytest.mark.parametrize("group", [1, 3])
def test_sample_stream_with_roulette(pt, sample_scene, group):
    """pt_stream_* with roulette on leaves exactly the sums of one pt_render per sample"""
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 64, 48)
    depth, seed, n = 8, 12, 9
    with pt.Context(g, m, cam) as a, pt.Context(g, m, cam) as b:
        for c in (a, b):
            c.set_russian_roulette(2)
        b.stream_begin(0, 0, depth, seed, group)
        for k in range(n):
            a.render(k, 1, depth, seed)
            mean, spp = b.stream_next()
            assert spp == k + 1 and same_bits(mean, a.download_mean(k + 1)), k
        b.stream_end()
        assert same_bits(b.download_sum(), a.download_sum())


def test_cudaRaytraceCore_roulette_switch_restarts_the_stream(pt, oracle, sample_scene):
    """compat.set_russian_roulette changes the estimator for the calls that follow: samples traced ahead with the old
    setting are dropped"""
    compat = importlib.import_module("project3-pathtracer_b200.compat")
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = with_resolution(sample_scene["camera"], 64, 64)
    rs = compat.RefScene([(g, cam)], m, iterations=4)
    compat.reset(); compat.set_trace_depth(8); compat.set_seed(6); compat.set_exit_on_error(False)
    call = lambda k: compat.cudaRaytraceCore(None, rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))  # noqa: E731
    on, off = oracle.make_scene(g, m, cam, roulette=1), oracle.make_scene(g, m, cam)
    want = np.zeros((64 * 64, 3), np.float32)
    try:
        with pytest.raises(ValueError):
            compat.set_russian_roulette(64)
        compat.set_russian_roulette(1)
        for k in (1, 2):
            call(k)
            oracle.render(on, k - 1, 1, 8, 6, sum_rgb=want)
        assert same_bits(rs.image, want / np.float32(2))
        compat.set_russian_roulette(0)  # sample 2 was traced ahead with roulette: it must not count
        call(3)
        oracle.render(off, 2, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(3), rtol=1e-6, atol=1e-6)
        compat.set_russian_roulette(1)
        call(4)
        oracle.render(on, 3, 1, 8, 6, sum_rgb=want)
        assert np.allclose(rs.image, want / np.float32(4), rtol=1e-6, atol=1e-6)
        assert compat.last_status() == 0
    finally:
        compat.set_russian_roulette(0)
        compat.reset()


def test_headless_driver_roulette(pt, tmp_path):
    """pt_render scene=scenes/sample.txt rr=K (reduced): the segments and image the C ABI renders"""
    from PIL import Image
    src = open(os.path.join(ROOT, "scenes", "sample.txt")).read()
    p = tmp_path / "sample.txt"
    p.write_text(re.sub(r"RES\s+\d+\s+\d+", "RES         96 64", src, count=1))
    g, m, cam, lens = pt.Scene(p).frame(0)
    exe = os.path.join(ROOT, "project3-pathtracer_b200", "pt_render")
    segs_seen = []
    for k in (2, 0):
        out = subprocess.check_output([exe, "scene=%s" % p, "spp=2", "depth=8", "seed=8", "rr=%d" % k,
                                       "out=%s" % (tmp_path / ("r%d.png" % k)), "json=1"], text=True)
        info = json.loads(out.strip().splitlines()[-1])
        with pt.Context(g, m, cam, lens) as c:
            c.set_russian_roulette(k)
            c.render(0, 2, 8, 8)
            want_sum = c.download_sum()
            _, segs, _ = c.counters()
        assert info["segments"] == int(segs)
        got8 = np.asarray(Image.open(info["file"]).convert("RGB"))
        assert (got8 == pt.image_to_rgb8(want_sum / np.float32(2), 96, 64)).all()
        segs_seen.append(int(segs))
    assert segs_seen[0] < segs_seen[1]
    assert subprocess.run([exe, "scene=%s" % p, "spp=1", "rr=64", "out=%s" % (tmp_path / "bad.png")],
                          capture_output=True).returncode != 0
