"""Scenes for the glossy-reflection tests (tests/test_oracle_glossy.py on the CPU, tests/test_gpu_glossy.py)."""
import numpy as np

from conftest import optics_scene
from medium_scenes import material, media_scene
from scenes_for_tests import build_geom, random_scene


def _glossy(m):
    """optics_scene's materials with its mirror sphere (material 3) glossy, a glossy wall material appended (index 9,
    for the back wall), and SPECEX on materials that must keep ignoring it: a diffuse one (1) and the glass sphere (4)"""
    m = np.concatenate([m, m[:1]])
    m[3]["specularExponent"] = 20.0
    m[9]["hasReflective"], m[9]["specularExponent"], m[9]["specularColor"] = 1.0, 60.0, [0.8, 0.8, 0.8]
    m[1]["specularExponent"] = 7.0
    m[4]["specularExponent"] = 30.0
    return m


def glossy_scene(pt, sample_scene):
    """the sample scene's geometry: a glossy sphere, a glossy back wall, glass, diffuse walls and the light"""
    g, m = optics_scene(pt, sample_scene)
    g = g.copy()
    g[1]["materialid"] = 9
    return g, _glossy(m)


def glossy_media_scene(pt, sample_scene):
    """glossy_scene with its glass turned into media (media_scene): glossy reflection and subsurface scattering together"""
    g, m = media_scene(pt, sample_scene)
    g = g.copy()
    g[1]["materialid"] = 9
    return g, _glossy(m)


def glossy_hierarchy_scene(pt, sample_scene, n=40):
    """n >= 33 random geoms (the hierarchy kernels), a third of them glossy, under the sample scene's light"""
    g, m = glossy_scene(pt, sample_scene)
    light = int(sample_scene["geoms"][8]["materialid"])
    gg = random_scene(pt, n, 11, extent=6.0, smin=0.3, smax=2.0)
    gg["materialid"] = np.array([3, 9, 0, 1, 2, 4])[np.arange(n) % 6]
    gg[n - 1] = build_geom(pt, 1, light, (0, 9, 0), (0, 0, 0), (5, 0.3, 5))
    return gg, m


def as_mirrors(m):
    """the same materials with SPECEX 0: every glossy reflector a perfect mirror"""
    m0 = m.copy()
    m0["specularExponent"] = 0
    return m0


def furnace(pt, camera, w=32, h=32, specex=8.0):
    """A closed box of emissive walls (RGB 1, EMITTANCE 1) around a glossy sphere (SPECRGB 0.5): a camera ray that meets a
    wall adds exactly 1.0, one that meets the sphere leaves it above its surface (the fold), reaches a wall and adds
    exactly 0.5."""
    mats = np.zeros(2, pt.MATERIAL_DTYPE)
    mats[0] = material(pt, emittance=1.0)
    mats[1] = material(pt, spec=(0.5, 0.5, 0.5))
    mats[1]["hasReflective"], mats[1]["specularExponent"] = 1.0, specex
    walls = [((0, -3, 0), (8, .2, 8)), ((0, 3, 0), (8, .2, 8)), ((-3, 0, 0), (.2, 8, 8)), ((3, 0, 0), (.2, 8, 8)),
             ((0, 0, -3), (8, 8, .2)), ((0, 0, 3), (8, 8, .2))]
    g = np.zeros(len(walls) + 1, pt.GEOM_DTYPE)
    for i, (t, s) in enumerate(walls):
        g[i] = build_geom(pt, 1, 0, t, (0, 0, 0), s)
    g[len(walls)] = build_geom(pt, 0, 1, (0, 0, -0.8), (0, 0, 0), (2.4, 2.4, 2.4))
    cam = camera.copy()
    cam["resolution"][0] = [w, h]
    cam["position"][0] = [0, 0, 2.6]
    cam["view"][0] = [0, 0, -1]
    cam["up"][0] = [0, 1, 0]
    cam["fov"][0] = [30, 30]
    return g, mats, cam
