"""Subsurface scattering in the C restatement (the specification the kernels follow bit for bit, DESIGN.md 4): the
reproducible log, the statistics of the free flight, a white furnace, the switch, and the frozen golden vectors.
CPU only."""
import json
import os
import sys

import numpy as np
import pytest
from scipy import integrate

from conftest import GOLD, ROOT, f32, same_bits, with_resolution
from medium_scenes import furnace, media_scene


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering (oracle/pt_oracle_medium.c)"""
    from oracle_medium import OracleMedium
    return OracleMedium()


def test_log_relative_error_on_every_free_flight_argument(oracle):
    """or_log against binary64 log on all 2^24 arguments 1 - k 2^-24 the renderer can pass (xf = k 2^-24): the free
    flight s = -log(1 - xf) / sigma_s with sigma_s = 1 and an infinite segment is -or_log itself"""
    worst, chunk = 0.0, 1 << 22
    for k0 in range(0, 1 << 24, chunk):
        k = np.arange(k0, k0 + chunk, dtype=np.float64)
        u = np.zeros((chunk, 3), np.float32)
        u[:, 2] = (k * 2.0 ** -24).astype(np.float32)
        _, s, _, _ = oracle.sample_medium(np.zeros((chunk, 3)), np.ones(chunk), np.full(chunk, np.inf), u)
        want = -np.log1p(-k * 2.0 ** -24)
        nz = want != 0
        assert (s[~nz] == 0).all()
        worst = max(worst, float((np.abs(s[nz] - want[nz]) / want[nz]).max()))
    assert worst <= 2.0 ** -22, worst
    assert oracle.log(1.0) == 0.0 and oracle.log(0.5) == np.float32(np.log(0.5))
    assert oracle.log(0.0) == -np.inf and oracle.log(-1.0) == -np.inf


def test_free_flight_statistics(oracle):
    n, sigma, t = 10 ** 6, 1.7, 0.9
    rng = np.random.default_rng(31)
    u = (rng.integers(0, 1 << 24, (n, 3)) * 2.0 ** -24).astype(np.float32)
    ab = np.tile(np.float32([0.3, 1.1, 0.0]), (n, 1))
    flag, s, dirs, w = oracle.sample_medium(ab, np.full(n, sigma), np.full(n, t), u)
    # P(scatter) = 1 - exp(-sigma t)
    p = 1 - np.exp(-sigma * t)
    assert abs(flag.mean() - p) <= 5 * np.sqrt(p * (1 - p) / n)
    # s given a scattering event: the exponential truncated to [0, t)
    m = int(flag.sum())
    dens = lambda x: sigma * np.exp(-sigma * x) / p  # noqa: E731
    mean = integrate.quad(lambda x: x * dens(x), 0, t)[0]
    var = integrate.quad(lambda x: x * x * dens(x), 0, t)[0] - mean ** 2
    assert abs(s[flag].mean() - mean) <= 5 * np.sqrt(var / m)
    assert (s[flag] < t).all() and (s[~flag] >= t).all()
    # directions uniform on the sphere: unit length, mean 0, E[z^2] = 1/3 (Var z^2 = 1/5 - 1/9)
    d = dirs[flag].astype(np.float64)
    assert np.abs(np.linalg.norm(d, axis=1) - 1).max() < 1e-6
    assert (np.abs(d.mean(0)) <= 5 * np.sqrt(1 / 3 / m)).all()
    assert abs((d[:, 2] ** 2).mean() - 1 / 3) <= 5 * np.sqrt(4 / 45 / m)
    assert not dirs[~flag].any()
    # weights: exactly calculateTransmission over s (scattered) or over the whole segment (passed through)
    assert same_bits(w[flag], oracle.transmission(ab[flag], s[flag]))
    assert same_bits(w[~flag], oracle.transmission(ab[~flag], np.full(n - m, t)))


def test_white_furnace(pt, oracle, sample_scene):
    """every boundary event leaves the throughput at exactly 1: every path that ends on a wall adds exactly 1.0, so pixel
    sums are integers and, at depth 64, nearly every path gets out of the medium"""
    w = h = 32
    spp, depth = 2, 64
    g, m, cam = furnace(pt, sample_scene["camera"], w, h)
    img, live, _ = oracle.render(oracle.make_scene(g, m, cam, subsurface=True), 0, spp, depth, 7)
    assert (img == np.round(img)).all()
    assert (img[:, 0] == img[:, 1]).all() and (img[:, 0] == img[:, 2]).all()
    paths = w * h * spp
    assert img[:, 0].sum() >= (1 - 1e-4) * paths
    _, live_glass, _ = oracle.render(oracle.make_scene(g, m, cam, subsurface=False), 0, spp, depth, 7)
    assert live.sum() > 1.5 * live_glass.sum()  # scattering happened: many more segments than through plain glass


def test_switch_changes_nothing_without_a_medium(pt, oracle, sample_scene):
    g, m = media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 48, 48)
    spp, depth, seed = 2, 8, 5

    def render(mats, sss):
        return oracle.render(oracle.make_scene(g, mats, cam, subsurface=sss), 0, spp, depth, seed)[:2]

    on_img, on_live = render(m, True)
    off_img, off_live = render(m, False)
    assert not same_bits(on_img, off_img)  # (the scene has media: the switch matters)
    # on, but RSCTCOEFF 0: no medium, the same image as off
    m0 = m.copy()
    m0["reducedScatterCoefficient"] = 0
    img, live = render(m0, True)
    assert same_bits(img, off_img) and (live == off_live).all()
    # off, SCATTER 1: the same image as SCATTER 0
    m1 = m.copy()
    m1["hasScatter"] = 0
    img, live = render(m1, False)
    assert same_bits(img, off_img) and (live == off_live).all()


def test_path_loop_without_media_is_the_restatement(pt, oracle, sample_scene):
    """or_render_sss with the switch off, and on a scene without media, is the unmodified restatement's render (the
    library built from oracle/pt_oracle.c alone) bit for bit, direct light sampling included"""
    from oracle_py import Oracle
    plain = Oracle()
    g, m = media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 48, 48)
    m_glass = m.copy()
    m_glass["hasScatter"] = 0
    for mats, sss in ((m, False), (m_glass, True)):
        for nee in (False, True):
            want, want_live, _ = plain.render(plain.make_scene(g, mats, cam, direct_lighting=nee), 0, 2, 6, 13)
            got, live, _ = oracle.render(oracle.make_scene(g, mats, cam, direct_lighting=nee, subsurface=sss), 0, 2, 6, 13)
            assert same_bits(got, want) and (live == want_live).all() and oracle.last_shadow_rays == plain.last_shadow_rays


def test_golden_medium_vectors_reproduce(oracle):
    with open(os.path.join(GOLD, "medium_vectors.json")) as f:
        gv = json.load(f)
    flag, s, dirs, w = oracle.sample_medium(f32(gv["absorption"]), f32(gv["scatter"]), f32(gv["distance"]), f32(gv["u"]))
    assert flag.astype(int).tolist() == gv["scattered"]
    assert 0 < sum(gv["scattered"]) < len(gv["scattered"])
    for got, key in ((s, "s"), (dirs, "direction"), (w, "weight")):
        assert same_bits(got.ravel(), f32(gv[key])), key


def test_cornell_sss_scene_is_generated():
    """scenes/gen_scenes.py writes the subsurface scene and leaves the other scene files as they are"""
    sys.path.insert(0, os.path.join(ROOT, "scenes"))
    import gen_scenes
    for name, text in (("cornell_sss.txt", gen_scenes.cornell_sss()), ("sample.txt", gen_scenes.sample_scene()),
                       ("cornell_glass_dof.txt", gen_scenes.cornell_glass_dof())):
        with open(os.path.join(ROOT, "scenes", name)) as f:
            assert f.read() == text, name
