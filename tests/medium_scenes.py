"""Scenes for the subsurface-scattering tests (tests/test_oracle_medium.py on the CPU, tests/test_gpu_subsurface.py)."""
import numpy as np

from conftest import optics_scene
from scenes_for_tests import build_geom, random_scene


def material(pt, color=(1, 1, 1), spec=(1, 1, 1), refr=0.0, ior=0.0, scatter=0.0, absorption=(0, 0, 0), rsct=0.0,
             emittance=0.0):
    m = np.zeros(1, pt.MATERIAL_DTYPE)[0]
    m["color"], m["specularColor"] = color, spec
    m["hasRefractive"], m["indexOfRefraction"] = refr, ior
    m["hasScatter"], m["absorptionCoefficient"], m["reducedScatterCoefficient"] = scatter, absorption, rsct
    m["emittance"] = emittance
    return m


def furnace(pt, camera, w=32, h=32):
    """A closed box of emissive walls (RGB 1, EMITTANCE 1) around a sphere of radius 1.6 that holds a non-absorbing medium
    of optical radius 2 (RSCTCOEFF 1.25) behind an index-matched boundary (REFRIOR 1, RGB 1, SPECRGB 1): every boundary
    event leaves the throughput at exactly 1, so every path that ends on a wall adds exactly 1.0."""
    mats = np.zeros(2, pt.MATERIAL_DTYPE)
    mats[0] = material(pt, emittance=1.0)
    mats[1] = material(pt, refr=1.0, ior=1.0, scatter=1.0, rsct=1.25)
    walls = [((0, -3, 0), (8, .2, 8)), ((0, 3, 0), (8, .2, 8)), ((-3, 0, 0), (.2, 8, 8)), ((3, 0, 0), (.2, 8, 8)),
             ((0, 0, -3), (8, 8, .2)), ((0, 0, 3), (8, 8, .2))]
    g = np.zeros(len(walls) + 1, pt.GEOM_DTYPE)
    for i, (t, s) in enumerate(walls):
        g[i] = build_geom(pt, 1, 0, t, (0, 0, 0), s)
    g[len(walls)] = build_geom(pt, 0, 1, (0, 0, -0.8), (0, 0, 0), (3.2, 3.2, 3.2))
    cam = camera.copy()
    cam["resolution"][0] = [w, h]
    cam["position"][0] = [0, 0, 2.6]
    cam["view"][0] = [0, 0, -1]
    cam["up"][0] = [0, 1, 0]
    cam["fov"][0] = [30, 30]
    return g, mats, cam


def media_scene(pt, sample_scene):
    """optics_scene with its glass sphere (material 4) and glass cube material (6) turned into media, one of them
    absorbing"""
    g, m = optics_scene(pt, sample_scene)
    m[4]["hasScatter"], m[4]["reducedScatterCoefficient"] = 1.0, 0.8
    m[4]["absorptionCoefficient"] = [0.05, 0.2, 0.4]
    m[6]["hasScatter"], m[6]["reducedScatterCoefficient"] = 1.0, 3.0
    return g, m


def media_hierarchy_scene(pt, sample_scene, n=40):
    """n >= 33 random geoms (the hierarchy kernels), a third of them media, under the sample scene's light"""
    g, m = media_scene(pt, sample_scene)
    light = int(sample_scene["geoms"][8]["materialid"])
    gg = random_scene(pt, n, 11, extent=6.0, smin=0.3, smax=2.0)
    gg["materialid"] = np.array([4, 6, 0, 1, 2, 3])[np.arange(n) % 6]
    gg[n - 1] = build_geom(pt, 1, light, (0, 9, 0), (0, 0, 0), (5, 0.3, 5))
    return gg, m
