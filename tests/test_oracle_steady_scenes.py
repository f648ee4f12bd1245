"""CPU checks of what tests/test_gpu_steady_state.py relies on in tests/steady_scenes.py: the copies of a geom are hit
often enough to force fallbacks and deferrals at volume, their tie-break shows in the image, the paths stay alive long
enough for the frame sizes, and each scene runs the kernels it is meant for."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from steady_scenes import (HIERARCHY_KEEP_DEPTH1, ROOM_KEEP_DEPTH4, hierarchy_side, room_side, steady_hierarchy,
                           steady_room, tickets_per_warp)


@pytest.fixture(scope="module")
def oracle():
    from oracle_roulette import OracleRoulette
    return OracleRoulette()


@pytest.fixture(scope="module", params=["room", "hierarchy"])
def scene(request, pt, sample_scene):
    """(name, geoms, materials, camera at 64x64, groups of exact copies)"""
    if request.param == "room":
        g, m, cam = steady_room(pt, sample_scene["camera"], 64, 64)
        return "room", g, m, cam, [[7, 8], [9, 10]]
    g, m, cam, twins, triplets = steady_hierarchy(pt, sample_scene["camera"], 64, 64)
    return "hierarchy", g, m, cam, twins + triplets


def _bvh_min_geoms():
    src = open(os.path.join(ROOT, "project3-pathtracer_b200", "csrc", "pt_api.cu")).read()
    return int(re.search(r"static const int kBvhMinGeoms = (\d+);", src).group(1))


def test_geom_counts_pick_the_kernels(scene):
    name, g, _, _, groups = scene
    if name == "room":
        assert len(g) < _bvh_min_geoms()
    else:
        assert len(g) >= _bvh_min_geoms()
        assert sum(len(x) == 2 for x in groups) >= 2 and sum(len(x) == 3 for x in groups) >= 2


def test_copies_are_exact_with_distinct_materials(scene):
    _, g, _, _, groups = scene
    for grp in groups:
        base = g[grp[0]]
        for i in grp[1:]:
            assert g[i]["type"] == base["type"]
            for f in ("transform", "inverseTransform"):
                assert (g[i][f].view(np.uint32) == base[f].view(np.uint32)).all()
        assert len({int(g[i]["materialid"]) for i in grp}) == len(grp)


def test_copies_are_hit_often(oracle, scene):
    """each group of copies is the closest hit of at least 1 % of the primary rays and of one diffuse bounce of them;
    the lowest index among the copies wins"""
    _, g, _, cam, groups = scene
    pix = np.arange(64 * 64, dtype=np.uint32)
    o, d = oracle.raygen(cam, (0.0, 0.0), 5, pix, np.zeros_like(pix))
    gid, _, p, nr = oracle.intersect_rays(g, o, d)
    assert (gid >= 0).all()  # a closed room
    rng = np.random.default_rng(3)
    ob = (p + nr * np.float32(2e-4)).astype(np.float32)
    db = rng.normal(size=ob.shape).astype(np.float32)
    db /= np.linalg.norm(db, axis=1, keepdims=True).astype(np.float32)
    flip = (db * nr).sum(1) < 0
    db[flip] = -db[flip]
    gid2, _, _, _ = oracle.intersect_rays(g, ob, db)
    for grp in groups:
        for ids in (gid, gid2):
            hit = np.isin(ids, grp)
            assert hit.mean() >= 0.01, (grp, hit.mean())
            assert (ids[hit] == grp[0]).all()


def test_swapping_copies_changes_the_image(oracle, scene):
    """the materials of a group's copies swapped: a renderer that broke the tie the other way would differ"""
    _, g, m, cam, groups = scene
    base, _, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=True), 0, 1, 3, 9)
    for grp in groups:
        g2 = g.copy()
        g2["materialid"][grp[0]], g2["materialid"][grp[-1]] = g["materialid"][grp[-1]], g["materialid"][grp[0]]
        img, _, _ = oracle.render(oracle.make_scene(g2, m, cam, direct_lighting=True), 0, 1, 3, 9)
        assert np.abs(img - base).sum(axis=1).astype(bool).mean() >= 0.005, grp


@pytest.mark.parametrize("nee,sss,gl,rr", [(False, False, False, 0), (True, True, True, 1), (True, True, True, 3)])
def test_paths_stay_alive(oracle, scene, nee, sss, gl, rr):
    """at least 80 % of the paths are alive at depth 4, and at least the shares the frame sizes are computed for"""
    name, g, m, cam, _ = scene
    _, live, _ = oracle.render(oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss, glossy=gl, roulette=rr),
                               0, 2, 8, 13)
    keep = live / np.float64(64 * 64 * 2)
    assert keep[4] >= 0.8, keep
    if name == "room":
        assert keep[4] >= ROOM_KEEP_DEPTH4, keep
    else:
        assert keep[1] >= HIERARCHY_KEEP_DEPTH1, keep


def test_frame_sizes_follow_the_sm_count():
    for sms in (1, 108, 132, 148, 160):
        w = room_side(sms)
        assert w % 32 == 0
        assert tickets_per_warp(w * w * ROOM_KEEP_DEPTH4, sms) >= 6
        assert tickets_per_warp((w - 32) ** 2 * ROOM_KEEP_DEPTH4, sms) < 6
        h = hierarchy_side(sms)
        assert h % 32 == 0 and h * h * 2 * HIERARCHY_KEEP_DEPTH1 >= 2 * 32 * sms * 1024
    assert room_side(148) == 2080 and hierarchy_side(148) == 2240
