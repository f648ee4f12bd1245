"""Glossy reflection in the C restatement (the specification the kernels follow bit for bit, DESIGN.md 4): the lobe's
distribution, its geometry and fold, the mirror limit, a furnace, the switch, the path loop against the subsurface one,
and the frozen golden vectors.  CPU only."""
import json
import os
import sys

import numpy as np
import pytest
from scipy import stats

from conftest import GOLD, ROOT, f32, same_bits, with_resolution
from glossy_scenes import as_mirrors, furnace, glossy_media_scene, glossy_scene

U_TOP = np.float32(1 - 2.0 ** -24)


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering and glossy reflection (oracle/pt_oracle_glossy.c)"""
    from oracle_glossy import OracleGlossy
    return OracleGlossy()


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def lobe_f64(normal, incident, exponent, u):
    """the lobe in binary64 (the same construction, no reproducibility tricks) -> (folded direction, unfolded direction,
    ns, frame-rule margin, sin of the lobe angle): entries whose |r.x| or |r.y| lie within 1e-5 of 1/sqrt(3) may pick the
    other frame axis"""
    n, d = normal.astype(np.float64), incident.astype(np.float64)
    ns = np.where((np.einsum("ij,ij->i", d, n) < 0)[:, None], n, -n)
    r = d - 2 * np.einsum("ij,ij->i", d, ns)[:, None] * ns
    third = 1 / np.sqrt(3)
    ax = np.where(np.abs(r[:, 0]) < third, 0, np.where(np.abs(r[:, 1]) < third, 1, 2))
    dnn = np.eye(3)[ax]
    p1 = _unit(np.cross(r, dnn))
    p2 = _unit(np.cross(r, p1))
    c = (1 - u[:, 0].astype(np.float64)) ** (1 / (exponent.astype(np.float64) + 1))
    s = np.sqrt(np.maximum(0, 1 - c * c))
    phi = 2 * np.pi * u[:, 1].astype(np.float64)
    g = r * c[:, None] + p1 * (np.cos(phi) * s)[:, None] + p2 * (np.sin(phi) * s)[:, None]
    dn = np.einsum("ij,ij->i", g, ns)
    folded = np.where((dn > 0)[:, None], g, g - 2 * dn[:, None] * ns)
    margin = np.minimum(np.abs(np.abs(r[:, 0]) - third), np.abs(np.abs(r[:, 1]) - third))
    return folded, g, ns, margin, s


def _golden():
    with open(os.path.join(GOLD, "glossy_vectors.json")) as f:
        gv = json.load(f)
    return gv, f32(gv["normal"]).reshape(-1, 3), f32(gv["incident"]).reshape(-1, 3), f32(gv["exponent"]), f32(gv["u"]).reshape(-1, 2)


def test_golden_glossy_vectors_reproduce(oracle):
    gv, n, d, e, u = _golden()
    got = oracle.sample_glossy(n, d, e, u)
    assert same_bits(got.ravel(), f32(gv["direction"]))
    # the set covers what it claims: every exponent at every incidence, u at both ends, and the fold
    groups = set(gv["group"])
    for ex in ("0.001", "1", "10", "100", "10000", "1e+30"):
        for inc in ("normal", "oblique", "grazing"):
            assert "%s/%s" % (ex, inc) in groups
    assert (u == 0).any(axis=0).all() and (u == U_TOP).any(axis=0).all()
    _, g_unfolded, ns, _, _ = lobe_f64(n, d, e, u)
    assert (np.einsum("ij,ij->i", g_unfolded, ns) < -1e-3).any()


@pytest.mark.parametrize("exponent", [0.5, 1.0, 10.0, 100.0, 1000.0])
def test_lobe_cosine_distribution(oracle, exponent):
    """normal incidence (r = ns, so nothing is folded): cos of the angle to r has the CDF c^(n+1) (KS test, 10^6 samples)"""
    m = 10 ** 6
    rng = np.random.default_rng(int(exponent * 10) + 1)
    u = (rng.integers(0, 1 << 24, (m, 2)) * 2.0 ** -24).astype(np.float32)
    n = np.tile(np.float32([0, 0, 1]), (m, 1))
    g = oracle.sample_glossy(n, -n, np.full(m, exponent, np.float32), u)
    c = g[:, 2].astype(np.float64)
    assert (c >= 0).all()
    p = stats.kstest(c, lambda x: np.clip(x, 0, 1) ** (exponent + 1)).pvalue
    assert p > 1e-3, p
    # the azimuth is uniform too: the tangential part's angle
    phi = np.arctan2(g[:, 1], g[:, 0])[c < 0.999]
    assert stats.kstest(phi, stats.uniform(loc=-np.pi, scale=2 * np.pi).cdf).pvalue > 1e-3


@pytest.mark.parametrize("cos_i", [1.0, 0.5, 0.05, 0.005])
def test_lobe_geometry_and_fold(oracle, cos_i):
    """unit length within 1e-6, never below the surface, and the binary64 construction (fold included) within 1e-5 -- plus
    what one rounding of c near 1 moves the azimuth circle, 2^-24 / sin(angle); the fold is taken at grazing incidence"""
    m = 200000
    rng = np.random.default_rng(int(cos_i * 1000))
    n = _unit(rng.normal(size=(m, 3)))
    t = _unit(np.cross(n, rng.normal(size=(m, 3))))
    d = _unit(-cos_i * n + np.sqrt(1 - cos_i * cos_i) * t).astype(np.float32)
    n = n.astype(np.float32)
    n[m // 2:] = -n[m // 2:]
    e = np.exp(rng.uniform(np.log(0.01), np.log(1e4), m)).astype(np.float32)
    u = (rng.integers(0, 1 << 24, (m, 2)) * 2.0 ** -24).astype(np.float32)
    g = oracle.sample_glossy(n, d, e, u)
    want, g_unfolded, ns, margin, sin_a = lobe_f64(n, d, e, u)
    assert np.abs(np.linalg.norm(g.astype(np.float64), axis=1) - 1).max() < 1e-6
    assert (np.einsum("ij,ij->i", g.astype(np.float64), ns) >= 0).all()
    ok = margin > 1e-5
    err = np.abs(g - want).max(axis=1)
    assert (err[ok] < 1e-5 + 2.0 ** -24 / np.maximum(sin_a[ok], 1e-12)).all()
    folded = (np.einsum("ij,ij->i", g_unfolded, ns) < -1e-4).sum()
    if cos_i <= 0.05:
        assert folded > m // 100
    if cos_i == 1.0:
        assert folded == 0


def test_huge_exponent_is_the_mirror(oracle):
    """SPECEX = 1e30: c = 1 and s = 0, so the sample is reflect(ns, d) bit for bit at non-grazing incidence"""
    m = 2000
    rng = np.random.default_rng(5)
    n = _unit(rng.normal(size=(m, 3))).astype(np.float32)
    d = _unit(rng.normal(size=(m, 3))).astype(np.float32)
    cos = np.abs(np.einsum("ij,ij->i", n.astype(np.float64), d))
    n, d = n[cos > 0.1], d[cos > 0.1]
    u = (rng.integers(0, 1 << 24, (len(n), 2)) * 2.0 ** -24).astype(np.float32)
    u[:4] = [[0, 0], [0, U_TOP], [U_TOP, 0], [U_TOP, U_TOP]]
    g = oracle.sample_glossy(n, d, np.full(len(n), 1e30, np.float32), u)
    ns = np.where((np.einsum("ij,ij->i", d, n) < 0)[:, None], n, -n)
    want = np.stack([oracle.reflect(ns[i], d[i]) for i in range(len(n))])
    assert same_bits(g, want)


def test_furnace(pt, oracle, sample_scene):
    """a glossy sphere of SPECRGB 0.5 in an emissive box: every sample adds exactly 1 (a wall) or 0.5 (the sphere, then a
    wall), so every pixel sum is spp - k/2 for the k samples that met the sphere"""
    spp = 4
    g, m, cam = furnace(pt, sample_scene["camera"], 48, 48)
    img, live, _ = oracle.render(oracle.make_scene(g, m, cam, glossy=True), 0, spp, 8, 3)
    assert (img[:, 0] == img[:, 1]).all() and (img[:, 0] == img[:, 2]).all()
    k = 2 * (spp - img[:, 0])
    assert (k == np.round(k)).all() and (k >= 0).all() and (k <= spp).all()
    assert (img[:, 0] == spp).sum() > 0 and (img[:, 0] == spp / 2).sum() > 0.2 * len(img)
    assert live[2] == 0  # no path lives beyond the wall after the sphere


def test_switch_changes_nothing_without_a_glossy_geom(pt, oracle, sample_scene):
    """on, with SPECEX only on materials that are not glossy reflectors (diffuse, glass, emissive), or with SPECEX 0: the
    image of the switch off"""
    g, m = glossy_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 48, 48)

    def render(mats, glossy):
        return oracle.render(oracle.make_scene(g, mats, cam, glossy=glossy), 0, 2, 8, 5)[:2]

    off_img, off_live = render(m, False)
    on_img, _ = render(m, True)
    assert not same_bits(on_img, off_img)  # (the scene has glossy geoms: the switch matters)
    m0 = as_mirrors(m)
    m0["specularExponent"][[1, 4, 8]] = 9.0  # diffuse, glass, light
    for mats, glossy in ((m0, True), (as_mirrors(m), True), (m, False)):
        img, live = render(mats, glossy)
        assert same_bits(img, off_img) and (live == off_live).all()


def test_path_loop_without_glossy_is_the_subsurface_loop(pt, oracle, sample_scene):
    """or_render_ext with glossy == 0 is or_render_sss bit for bit, subsurface on and off, direct light sampling included"""
    g, m = glossy_media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 48, 48)
    for sss in (False, True):
        for nee in (False, True):
            sc = oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss)
            want, want_live, _ = oracle.render(sc, 0, 2, 6, 13, path_loop="sss")
            shadow = oracle.last_shadow_rays
            got, live, _ = oracle.render(sc, 0, 2, 6, 13)
            assert same_bits(got, want) and (live == want_live).all() and oracle.last_shadow_rays == shadow


def test_cornell_glossy_scene_is_generated():
    """scenes/gen_scenes.py writes the glossy scene and leaves the other scene files as they are"""
    sys.path.insert(0, os.path.join(ROOT, "scenes"))
    import gen_scenes
    for name, text in (("cornell_glossy.txt", gen_scenes.cornell_glossy()), ("cornell_sss.txt", gen_scenes.cornell_sss()),
                       ("sample.txt", gen_scenes.sample_scene()), ("cornell_glass_dof.txt", gen_scenes.cornell_glass_dof()),
                       ("sample_4k.txt", gen_scenes.sample_scene((3840, 2160), 16384))):
        with open(os.path.join(ROOT, "scenes", name)) as f:
            assert f.read() == text, name
