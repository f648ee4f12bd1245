"""GPU parity of the persistent bounce kernels in the state they run in at production sizes (DESIGN.md 6): frames sized
from the SM count so that every warp takes many tickets per depth (k_bounce, k_bounce_q) and the hierarchy kernel takes
full 1 024-path pools (k_bounce_bvh), with exact-scan fallbacks, second-candidate retries and deferred exact traversals
forced at volume by exact copies of geoms (tests/steady_scenes.py).  Each configuration is rendered once by the oracle
and compared with every GPU run of it: per-depth live counts identical, the image bit-identical without direct light
sampling (a pixel gets at most two contributions, so the order of the atomic additions cannot matter), with it the
shadow-ray count identical and the image within 1e-5 of each pixel's sum.  After each GPU render the precondition
(tickets per warp at each depth, fallback and retry volumes) is printed and asserted: a run that misses it checks
nothing."""
import itertools
import time

import numpy as np
import pytest

from conftest import same_bits, with_resolution
from steady_scenes import (POOL_PATHS, bounce_warps, hierarchy_side, room_side, steady_hierarchy, steady_room,
                           tickets_per_warp)

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5
ROOM_DEPTH = 8
HIERARCHY_DEPTH = 4
SPP = 2


@pytest.fixture(scope="module")
def oracle():
    from oracle_roulette import OracleRoulette
    return OracleRoulette()


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _oracle(oracle, g, m, cam, depth, seed, nee=False, sss=False, gl=False, rr=0):
    t0 = time.time()
    want, live, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss, glossy=gl,
                                                    roulette=rr), 0, SPP, depth, seed)
    print("  oracle: %d segments in %.1f s" % (int(live.sum()), time.time() - t0))
    return want, live, oracle.last_shadow_rays


def _gpu(pt, g, m, cam, depth, seed, nee=False, sss=False, gl=False, rr=0, policy=0, wavefront_paths=None, band=None):
    with pt.Context(g, m, cam) as c:
        c.set_kernel_policy(policy)
        c.set_direct_lighting(nee)
        c.set_subsurface(sss)
        c.set_glossy(gl)
        c.set_russian_roulette(rr)
        if wavefront_paths is not None:
            c.set_wavefront_paths(wavefront_paths)
        if band is not None:
            c.set_band_pixels(band)
        c.render(0, SPP, depth, seed)
        img = c.download_sum()
        _, segs, live = c.counters()
        return dict(img=img, segs=int(segs), live=live[:depth].astype(np.int64), shadow=c.shadow_rays()[0],
                    fallbacks=c.filter_stats(), retries=c.filter_retries())


def _report(tag, run, sms, wavefronts):
    t = tickets_per_warp(run["live"], sms, wavefronts)
    print("  %s: tickets per warp by depth %s; fallbacks %d (%.2f %% of %d segments, %.1f per warp), retries %d (%.2f %%)"
          % (tag, np.array2string(t, precision=1), run["fallbacks"], 100.0 * run["fallbacks"] / run["segs"], run["segs"],
             run["fallbacks"] / bounce_warps(sms), run["retries"], 100.0 * run["retries"] / run["segs"]))
    return t


def _compare(tag, run, want, want_live, want_shadow, nee, width):
    got, live = run["img"], run["live"]
    bad = [d for d in range(len(want_live)) if live[d] != int(want_live[d])]
    assert not bad, "%s: live counts differ at depths %s: gpu %s, oracle %s" % (
        tag, bad, [int(live[d]) for d in bad], [int(want_live[d]) for d in bad])
    if nee:
        assert run["shadow"] == want_shadow, (tag, run["shadow"], want_shadow)
        diff = ~np.isclose(got, want, rtol=SUM_TOL, atol=SUM_TOL).all(axis=1)
    else:
        diff = (got.view(np.uint32) != want.view(np.uint32)).any(axis=1)
    idx = np.flatnonzero(diff)
    assert idx.size == 0, "%s: %d pixels differ, first: %s" % (tag, idx.size, "; ".join(
        "(%d, %d) gpu %s oracle %s" % (i % width, i // width, got[i].tolist(), want[i].tolist()) for i in idx[:8]))


def _variants():
    """all 16 launch variants of the bounce kernels; roulette from depth 1 in half of the roulette-on ones and from
    depth 3 (the instantiation changes mid-wavefront) in the other half"""
    for nee, sss, gl, rr in itertools.product((False, True), repeat=4):
        k = (1 if (nee ^ sss ^ gl) == 0 else 3) if rr else 0
        yield pytest.param(nee, sss, gl, k, id="nee%d-sss%d-glossy%d-rr%d" % (nee, sss, gl, k))


@pytest.mark.parametrize("nee,sss,gl,rr", list(_variants()))
def test_room_every_variant_at_full_occupancy(pt, oracle, sample_scene, sms, nee, sss, gl, rr):
    """steady_room at room_side(SMs)^2 x 2 spp, depth 8: k_bounce_q (policy 1, one wavefront per sample, two in flight
    on both slots) and the fused k_bounce (policy 2, both samples in one wavefront)"""
    side = room_side(sms)
    g, m, cam = steady_room(pt, sample_scene["camera"], side, side)
    npix = side * side
    print("\nroom %dx%d x %d spp on %d SMs, %s" % (side, side, SPP, sms, dict(nee=nee, sss=sss, glossy=gl, rr=rr)))
    want, want_live, want_shadow = _oracle(oracle, g, m, cam, ROOM_DEPTH, 31, nee, sss, gl, rr)
    for policy, wavefronts, wf_paths in ((1, 2, npix), (2, 1, None)):
        run = _gpu(pt, g, m, cam, ROOM_DEPTH, 31, nee, sss, gl, rr, policy=policy, wavefront_paths=wf_paths, band=npix)
        tag = "policy %d" % policy
        t = _report(tag, run, sms, wavefronts)
        assert (t[1:5] >= 6).all(), (tag, t)
        if not nee:
            assert run["fallbacks"] >= 0.01 * run["segs"] and run["fallbacks"] >= 10 * bounce_warps(sms), tag
        _compare(tag, run, want, want_live, want_shadow, nee, side)


@pytest.mark.parametrize("nee,sss,gl,rr", [(False, False, False, 0), (False, True, True, 1), (True, False, False, 0),
                                           (True, True, True, 2)],
                         ids=["off", "sss-glossy-rr1", "nee", "all-rr2"])
def test_hierarchy_full_pools(pt, oracle, sample_scene, sms, nee, sss, gl, rr):
    """steady_hierarchy at hierarchy_side(SMs)^2 x 2 spp in one wavefront, depth 4: k_raygen_wf and k_bounce_bvh with
    full pools at depths 0 and 1, second-candidate retries and deferred exact traversals in most warps"""
    side = hierarchy_side(sms)
    g, m, cam, _, _ = steady_hierarchy(pt, sample_scene["camera"], side, side)
    print("\nhierarchy (%d geoms) %dx%d x %d spp on %d SMs, %s" % (len(g), side, side, SPP, sms,
                                                                  dict(nee=nee, sss=sss, glossy=gl, rr=rr)))
    want, want_live, want_shadow = _oracle(oracle, g, m, cam, HIERARCHY_DEPTH, 41, nee, sss, gl, rr)
    run = _gpu(pt, g, m, cam, HIERARCHY_DEPTH, 41, nee, sss, gl, rr, band=side * side)
    _report("hierarchy", run, sms, 1)
    assert (run["live"][:2] >= 2 * bounce_warps(sms) * POOL_PATHS).all(), run["live"]
    assert run["retries"] >= 0.01 * run["segs"]
    assert run["fallbacks"] >= 0.01 * run["segs"] and run["fallbacks"] >= 64 * bounce_warps(sms)
    _compare("hierarchy", run, want, want_live, want_shadow, nee, side)


def test_strong_shape_automatic_bands(pt, oracle, sample_scene, sms):
    """the sample scene at 3840x2160 x 2 spp, depth 8, policy 0: automatic 1 Mi-pixel bands, wavefronts alternating
    between both slots"""
    cam = with_resolution(sample_scene["camera"], 3840, 2160)
    g, m = sample_scene["geoms"], sample_scene["materials"]
    print("\nsample scene 3840x2160 x %d spp on %d SMs" % (SPP, sms))
    want, want_live, _ = _oracle(oracle, g, m, cam, ROOM_DEPTH, 53)
    run = _gpu(pt, g, m, cam, ROOM_DEPTH, 53)
    _report("strong, per 1 Mi-pixel band", run, sms, 3840 * 2160 / (1 << 20))
    _compare("strong", run, want, want_live, 0, False, 3840)


def test_sample_stream_at_shim_size(pt, oracle, sample_scene):
    """800x800 (the shim's frame): a 2-sample base, then 17 streamed samples in groups of 8 -- more than two groups, so
    the groups alternate and refill; each mean equals the oracle's sample-by-sample sum over its divisor"""
    cam = with_resolution(sample_scene["camera"], 800, 800)
    g, m = sample_scene["geoms"], sample_scene["materials"]
    depth, seed, n = 8, 67, 17
    sc = oracle.make_scene(g, m, cam)
    want = np.zeros((800 * 800, 3), np.float32)
    oracle.render(sc, 0, 2, depth, seed, sum_rgb=want)
    with pt.Context(g, m, cam) as c:
        c.render(0, 2, depth, seed)
        c.stream_begin(2, 2, depth, seed, 8)
        for k in range(1, n + 1):
            oracle.render(sc, 1 + k, 1, depth, seed, sum_rgb=want)
            mean, spp = c.stream_next()
            assert spp == 2 + k
            assert same_bits(mean, want / np.float32(2 + k)), k
        c.stream_end()
        assert same_bits(c.download_sum(), want)
