"""Russian roulette in the C restatement (the specification the kernels follow bit for bit, DESIGN.md 4): the step itself,
the path loop against the glossy one while roulette cannot run, white scenes, the segments it saves, and unbiasedness.
CPU only."""
import itertools

import numpy as np
import pytest

from conftest import same_bits, with_resolution
from glossy_scenes import glossy_media_scene
from roulette_scenes import batch_means, closed_room, white, within_standard_errors

SWITCHES = list(itertools.product([False, True], repeat=3))  # (direct lighting, subsurface, glossy)


@pytest.fixture(scope="module")
def oracle():
    """the C restatement extended by subsurface scattering, glossy reflection and Russian roulette
    (oracle/pt_oracle_roulette.c)"""
    from oracle_roulette import OracleRoulette
    return OracleRoulette()


def test_roulette_step(oracle):
    """m >= 1: no draw, bits kept; m == 0: always ends; a survivor is divided by q = ceil(m 2^24) 2^-24, exactly"""
    thr = np.array([1.0, 0.25, np.float32(0.1)], np.float32)
    ok, t = oracle.roulette(7, 3, 1, 2, thr)
    assert ok and same_bits(t, thr)
    for s in range(64):
        assert oracle.roulette(7, s, 0, 2, [0, 0, 0])[0] is False
    m = np.float32(0.3)
    q = np.float32(np.ceil(np.float64(m) * 2 ** 24) * 2.0 ** -24)
    thr = np.array([0.1, m, 0.2], np.float32)
    out = [oracle.roulette(9, p, 0, 5, thr) for p in range(4000)]
    alive = [t for ok, t in out if ok]
    assert 0.25 < len(alive) / len(out) < 0.35
    for t in alive:
        assert same_bits(t, thr / q)
    for ok, t in out:
        if not ok:
            assert same_bits(t, thr)


def _scene(oracle, g, m, cam, switches, k):
    nee, sss, gl = switches
    return oracle.make_scene(g, m, cam, direct_lighting=nee, subsurface=sss, glossy=gl, roulette=k)


@pytest.mark.parametrize("switches", SWITCHES)
def test_off_and_out_of_reach_are_the_glossy_loop(pt, oracle, sample_scene, switches):
    """k = 0 and k >= max_depth - 1 give or_render_ext bit for bit, with every combination of the other switches"""
    g, m = glossy_media_scene(pt, sample_scene)
    cam = with_resolution(sample_scene["camera"], 40, 40)
    depth = 8
    want, want_live, _ = oracle.render(_scene(oracle, g, m, cam, switches, 0), 0, 2, depth, 5, path_loop="ext")
    for k in (0, depth - 1, depth, 63):
        got, live, _ = oracle.render(_scene(oracle, g, m, cam, switches, k), 0, 2, depth, 5)
        assert same_bits(got, want) and live.tolist() == want_live.tolist(), k
    got, live, _ = oracle.render(_scene(oracle, g, m, cam, switches, 1), 0, 2, depth, 5)
    assert live.sum() < want_live.sum()


@pytest.mark.parametrize("switches", [(False, False, False), (True, False, True)])
def test_white_scene_is_never_touched(pt, oracle, sample_scene, switches):
    """RGB and SPECRGB 1, no ABSCOEFF: the throughput never falls below 1, so any k renders what roulette off renders"""
    g, m = glossy_media_scene(pt, sample_scene)
    m = white(m)
    cam = with_resolution(sample_scene["camera"], 40, 40)
    want, want_live, _ = oracle.render(_scene(oracle, g, m, cam, switches, 0), 0, 2, 10, 8, path_loop="ext")
    for k in (1, 2, 5):
        got, live, _ = oracle.render(_scene(oracle, g, m, cam, switches, k), 0, 2, 10, 8)
        assert same_bits(got, want) and live.tolist() == want_live.tolist(), k


def test_roulette_traces_fewer_segments(pt, oracle, sample_scene):
    """albedo below 1: fewer segments from depth k + 1 on, the same up to depth k"""
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = with_resolution(sample_scene["camera"], 48, 48)
    _, off, _ = oracle.render(oracle.make_scene(g, m, cam), 0, 4, 16, 2)
    for k in (1, 3):
        _, on, _ = oracle.render(oracle.make_scene(g, m, cam, roulette=k), 0, 4, 16, 2)
        assert on[:k + 1].tolist() == off[:k + 1].tolist()
        assert on.sum() < off.sum() and (on <= off).all()


@pytest.mark.parametrize("nee", [False, True])
def test_unbiased(pt, oracle, sample_scene, nee):
    """a closed diffuse room with a light at depth 16: the mean of batched renders with roulette from depth 1 agrees with
    roulette off within 4 combined standard errors"""
    g, m, cam = closed_room(pt, sample_scene["camera"])

    def run(k):
        sc = oracle.make_scene(g, m, cam, direct_lighting=nee, roulette=k)
        return batch_means(lambda first, spp: oracle.render(sc, first, spp, 16, 31)[0], 24, 4)

    off, on = run(0), run(1)
    ok, a, b, se = within_standard_errors(on, off)
    assert ok, (a, b, se)
