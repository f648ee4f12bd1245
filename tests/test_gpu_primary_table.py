"""Depth 0's closest hit with the per-pixel primary-ray table (csrc/pt_kernels.cuh: k_primary_table, primary_hit) must
return the exact scan's answer bit for bit: the table's candidate first, then the filter, for the primary rays
pt_raygen makes.  Also: the table decides most primary rays of the sample scene, and without its margin (filter scale 0)
the rays it decides do go wrong at edges -- so the comparison can fail."""
import numpy as np
import pytest

from conftest import with_resolution
from scenes_for_tests import all_scenes, build_geom, random_scene, touching_scene

pytestmark = pytest.mark.gpu

SEED = 1234
MIN_DECIDED = 0.85  # measured on a B200: 0.893 (DESIGN.md 3a "primary rays")


def _cam(pt, w, h, pos, view, up=(0, 1, 0), fovy=45.0):
    cam = np.zeros(1, pt.CAMERA_DTYPE)
    fovx = np.degrees(np.arctan(np.tan(np.radians(fovy)) * w / h))
    cam["resolution"], cam["position"], cam["view"], cam["up"], cam["fov"] = (w, h), pos, view, up, (fovx, fovy)
    return cam


def _geoms(gs):
    g = np.zeros(len(gs), gs[0].dtype)
    for i, x in enumerate(gs):
        g[i] = x
    return g


def _check(pt, ctx, npix, spp, first_sample=0):
    """every pixel x spp samples: primary_hit == raygen + exact scan, bit for bit; returns the decided flags"""
    pixel = np.tile(np.arange(npix, dtype=np.uint32), spp)
    sample = np.repeat(np.arange(first_sample, first_sample + spp, dtype=np.uint32), npix)
    gid, t, p, nr, dec = ctx.primary_hit(SEED, pixel, sample)
    o, d = ctx.raygen(SEED, pixel, sample)
    wid, wt, wp, wn = ctx.intersect(o, d, mode=pt.HIT_EXACT_SCAN)
    hit = wid >= 0
    assert (gid == wid).all(), int((gid != wid).sum())
    assert (t.view(np.uint32) == wt.view(np.uint32)).all()
    assert (p[hit].view(np.uint32) == wp[hit].view(np.uint32)).all()
    assert (nr[hit].view(np.uint32) == wn[hit].view(np.uint32)).all()
    return dec


def test_sample_scene_full_frame(pt, sample_scene):
    """the bench's own frame, 800 x 800 x 16 samples; the table settles most primary rays"""
    g, m, cam = sample_scene["geoms"], sample_scene["materials"], sample_scene["camera"]
    with pt.Context(g, m, cam) as ctx:
        assert ctx.primary_table_info()[0]
        dec = _check(pt, ctx, ctx.npix, 16)
    assert dec.mean() >= MIN_DECIDED, dec.mean()


@pytest.mark.parametrize("w,h", [(1, 1), (7, 5)])
def test_huge_footprints(pt, sample_scene, w, h):
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = with_resolution(sample_scene["camera"], w, h)
    with pt.Context(g, m, cam) as ctx:
        _check(pt, ctx, w * h, 4096)


@pytest.mark.parametrize("fovy", [1.0, 80.0])
def test_narrow_and_wide_fov(pt, sample_scene, fovy):
    g, m = sample_scene["geoms"], sample_scene["materials"]
    cam = sample_scene["camera"].copy()
    cam = with_resolution(cam, 96, 96)
    cam["fov"][0] = [fovy, fovy]
    with pt.Context(g, m, cam) as ctx:
        _check(pt, ctx, ctx.npix, 64)


def test_special_scenes(pt, sample_scene):
    """an eye 1e-3 from a thin wall, an eye inside a sphere, touching spheres and wall corners, a tiny far sphere"""
    m = sample_scene["materials"]
    wall = [build_geom(pt, 1, 0, (0, 0, 0), (0, 0, 0), (6, 6, 0.02)), build_geom(pt, 0, 1, (1, 0.5, -2), (0, 0, 0), (1, 1, 1)),
            build_geom(pt, 1, 0, (0, -3, 0), (0, 0, 0), (6, 0.02, 6))]
    cases = [
        (_geoms(wall), _cam(pt, 64, 48, (0.3, 0.2, 0.011), (0.2, 0.1, -1))),     # looking into the wall from 1e-3
        (_geoms(wall), _cam(pt, 64, 48, (0.3, 0.2, 0.011), (1, 0, -0.001))),    # ... and along it
        (_geoms([build_geom(pt, 0, 0, (0, 0, 0), (0, 0, 0), (8, 8, 8)), build_geom(pt, 1, 1, (0.5, 0, 0.5), (0, 20, 0), (0.5, 0.5, 0.5)),
                 build_geom(pt, 0, 1, (-1, 0.5, 1), (0, 0, 0), (1, 1, 1))]),
         _cam(pt, 64, 48, (0.3, 0.2, -0.1), (0.3, -0.2, 1))),                    # eye inside a sphere
        (touching_scene(pt), _cam(pt, 64, 48, (6, 5, 7), (-6, -3, -7))),        # touching spheres, stacked cubes, corners
        (_geoms([build_geom(pt, 1, 0, (0, 0, 0), (0, 0, 0), (1, 1, 1)), build_geom(pt, 1, 0, (1, 0, 0), (0, 0, 0), (1, 1, 1)),
                 build_geom(pt, 1, 0, (0.5, 1, 0), (0, 0, 0), (2, 1, 1)), build_geom(pt, 0, 0, (1.5, 0.5, 0.5), (0, 0, 0), (1, 1, 1))]),
         _cam(pt, 64, 48, (3, 3, 4), (-2.5, -2.4, -4))),                        # wall corners
        (_geoms([build_geom(pt, 0, 0, (0, 0, -100), (0, 0, 0), (0.01, 0.01, 0.01)), build_geom(pt, 1, 0, (0, 0, -150), (0, 0, 0), (50, 50, 1))]),
         _cam(pt, 64, 48, (0, 0, 0), (0, 0, -1), fovy=0.05)),                   # a tiny far sphere
    ]
    for i, (g, cam) in enumerate(cases):
        with pt.Context(g, m, cam) as ctx:
            assert ctx.primary_table_info()[0], i
            _check(pt, ctx, ctx.npix, 64)


@pytest.mark.parametrize("scene", ["sample", "aniso100", "offset1e4", "touching", "mixed20"])
def test_random_pinhole_cameras(pt, scene):
    """every filter class (uniform and other spheres, axis-aligned and rotated cubes) under random pinhole cameras"""
    scenes = all_scenes(pt)
    if scene == "mixed20":
        g = random_scene(pt, 20, 7, extent=6.0, smin=0.3, smax=3.0, aniso=3.0)
        g = np.concatenate([g, scenes["sample"][0]])
        m = scenes["sample"][1]
    else:
        g, m, _ = scenes[scene]
    c = np.array([x["transform"].reshape(4, 4)[:3, 3] for x in g], np.float64)
    lo, hi = c.min(0) - 3, c.max(0) + 3
    rng = np.random.default_rng(sum(map(ord, scene)))
    for k in range(6):
        pos = rng.uniform(lo, hi)
        target = c[rng.integers(len(c))] + rng.normal(size=3)
        cam = _cam(pt, 48, 40, pos, target - pos, up=rng.normal(size=3), fovy=float(rng.uniform(5, 60)))
        with pt.Context(g, m, cam) as ctx:
            assert ctx.primary_table_info()[0], (scene, k)
            _check(pt, ctx, ctx.npix, 32, first_sample=100 * k)


def test_no_margin_goes_wrong(pt, sample_scene):
    """filter scale 0 shrinks the footprint bound to nothing: the table then answers for the central ray only, and rays
    it decides near silhouettes get a wrong closest hit.  (The filter's own mismatches at scale 0 are not counted.)"""
    g, m, cam = sample_scene["geoms"], sample_scene["materials"], sample_scene["camera"]
    with pt.Context(g, m, cam) as ctx:
        npix = ctx.npix
        pixel = np.tile(np.arange(npix, dtype=np.uint32), 4)
        sample = np.repeat(np.arange(4, dtype=np.uint32), npix)
        o, d = ctx.raygen(SEED, pixel, sample)
        wid, wt, _, _ = ctx.intersect(o, d, mode=pt.HIT_EXACT_SCAN)
        ctx.set_filter_scale(0.0)
        gid, t, _, _, dec = ctx.primary_hit(SEED, pixel, sample)
        bad = dec & ((gid != wid) | (t.view(np.uint32) != wt.view(np.uint32)))
        assert bad.sum() > 0
        ctx.set_filter_scale(1.0)
        gid, t, _, _, dec = ctx.primary_hit(SEED, pixel, sample)
        assert (gid == wid).all() and (t.view(np.uint32) == wt.view(np.uint32)).all()


def test_table_only_where_it_applies(pt, sample_scene):
    """no table for a thin-lens camera or a scene of the hierarchy; a scene update switches it off and on again"""
    g, m, cam = sample_scene["geoms"], sample_scene["materials"], with_resolution(sample_scene["camera"], 32, 32)
    with pt.Context(g, m, cam, lens=(0.2, 8.0)) as ctx:
        assert not ctx.primary_table_info()[0]
    big = np.concatenate([random_scene(pt, 40, 3, extent=4.0, smin=0.1, smax=0.5), g])
    with pt.Context(big, m, cam) as ctx:
        assert not ctx.primary_table_info()[0]
        with pytest.raises(pt.PtError):
            ctx.primary_hit(SEED, [0], [0])
    with pt.Context(g, m, cam) as ctx:
        assert ctx.primary_table_info()[0]
        ctx.update_scene(g, m, cam, lens=(0.2, 8.0))
        assert not ctx.primary_table_info()[0]
        ctx.update_scene(g, m, cam)
        assert ctx.primary_table_info()[0]


def test_render_launches_unchanged_and_fallbacks_rare(pt, sample_scene):
    """the table build is not a render launch; a render's fallbacks stay rare"""
    g, m, cam = sample_scene["geoms"], sample_scene["materials"], with_resolution(sample_scene["camera"], 200, 200)
    with pt.Context(g, m, cam) as ctx:
        n0 = ctx.launch_count()
        ctx.set_filter_scale(1.0)  # rebuilds filter and table
        assert ctx.launch_count() == n0
        ctx.render(0, 8, 8, 7)
        _, segs, _ = ctx.counters()
        assert ctx.filter_stats() / segs < 0.01
