"""Scenes for the Russian-roulette tests (tests/test_oracle_roulette.py on the CPU, tests/test_gpu_roulette.py)."""
import numpy as np

from medium_scenes import material
from scenes_for_tests import build_geom


def white(m):
    """the same materials with RGB and SPECRGB 1 and no ABSCOEFF: no event lowers a path's throughput below 1, so the
    roulette never draws"""
    w = m.copy()
    w["color"] = 1.0
    w["specularColor"] = 1.0
    w["absorptionCoefficient"] = 0.0
    return w


def closed_room(pt, camera, w=24, h=24, albedo=0.7):
    """a closed box of diffuse walls (RGB `albedo`) with an emissive panel under its ceiling and a diffuse sphere: every
    path stays in the room until it reaches the light or runs out of depth"""
    mats = np.zeros(3, pt.MATERIAL_DTYPE)
    mats[0] = material(pt, color=(albedo, albedo * 0.9, albedo * 0.8))
    mats[1] = material(pt, color=(1, 1, 1), emittance=4.0)
    mats[2] = material(pt, color=(0.5, 0.8, 0.6))
    walls = [((0, -3, 0), (8, .2, 8)), ((0, 3, 0), (8, .2, 8)), ((-3, 0, 0), (.2, 8, 8)), ((3, 0, 0), (.2, 8, 8)),
             ((0, 0, -3), (8, 8, .2)), ((0, 0, 3), (8, 8, .2))]
    g = np.zeros(len(walls) + 2, pt.GEOM_DTYPE)
    for i, (t, s) in enumerate(walls):
        g[i] = build_geom(pt, 1, 0, t, (0, 0, 0), s)
    g[len(walls)] = build_geom(pt, 1, 1, (0, 2.8, 0), (0, 0, 0), (2, .1, 2))
    g[len(walls) + 1] = build_geom(pt, 0, 2, (0.8, -1.8, -0.8), (0, 0, 0), (2, 2, 2))
    cam = camera.copy()
    cam["resolution"][0] = [w, h]
    cam["position"][0] = [0, 0, 2.6]
    cam["view"][0] = [0, 0, -1]
    cam["up"][0] = [0, 1, 0]
    cam["fov"][0] = [35, 35]
    return g, mats, cam


def batch_means(render, n_batches, spp):
    """mean pixel value of each of n_batches renders of spp samples over disjoint sample ranges: render(first, spp) ->
    the (npix, 3) sum"""
    return np.array([float(render(b * spp, spp).astype(np.float64).mean()) / spp for b in range(n_batches)])


def within_standard_errors(a, b, k=4.0):
    """|mean(a) - mean(b)| <= k combined standard errors of the two batch means"""
    se = np.sqrt(a.var(ddof=1) / a.size + b.var(ddof=1) / b.size)
    return abs(a.mean() - b.mean()) <= k * se, a.mean(), b.mean(), se
