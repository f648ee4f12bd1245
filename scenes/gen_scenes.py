#!/usr/bin/env python
"""Writes the scene files of the BASELINE.json configs in the reference's text format (SURVEY.md appendix A).

  sample.txt             configs 0/1: the same materials, camera and objects as the reference's
                         data/scenes/sampleScene.txt (values re-stated in the tables below, file text generated here;
                         tests/test_scene_loader.py checks that it parses to the same structs, bit for bit, as the
                         reference loader's parse of the reference's own file, tests/golden/ref_vectors.json)
  cornell_glass_dof.txt  config 2: closed Cornell box, two glass spheres, a mirror sphere, a glass cube, an emissive
                         panel, thin lens (LENS block), 1920x1080, 4096 spp, 12 bounces.  Authored without rotations
                         (axis-aligned slabs are scaled instead), so it means the same under the reference's radian
                         ROTAT quirk (SURVEY.md D1).
  sample_4k.txt          config 4: sample scene at 3840x2160, 16384 iterations
  cornell_sss.txt        subsurface scattering (pt_set_subsurface / pt_render sss=1): a closed room with a sphere and a
                         cube of the sample scene's material 5 coefficients (REFRIOR 2.2, ABSCOEFF .02 5.1 5.7,
                         RSCTCOEFF 13) with SCATTER 1 -- and RGB 1 1 1, since the sample's RGB 0 0 0 would stop every
                         path that refracts into them
  cornell_glossy.txt     glossy reflection (pt_set_glossy / pt_render glossy=1): the closed room of cornell_sss.txt with
                         three glossy spheres (SPECEX 10, 100, 1000), a glossy back wall (SPECEX 30) and a perfect
                         mirror sphere (SPECEX 0) for contrast
  procedural(n, seed)    config 3: n spheres/cubes, i.i.d. type, centre, scale, rotation (radians) and material from a
                         fixed seed; written on demand (python scenes/gen_scenes.py --procedural 10000 out.txt)
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# (RGB, SPECEX, SPECRGB, REFL, REFR, REFRIOR, SCATTER, ABSCOEFF, RSCTCOEFF, EMITTANCE)
SAMPLE_MATERIALS = [
    ((1, 1, 1), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),            # 0 white diffuse
    ((.63, .06, .04), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),      # 1 red diffuse
    ((.15, .48, .09), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),      # 2 green diffuse
    ((.63, .06, .04), 0, (1, 1, 1), 0, 0, 2, 0, (0, 0, 0), 0, 0),      # 3 red glossy
    ((1, 1, 1), 0, (1, 1, 1), 0, 0, 2, 0, (0, 0, 0), 0, 0),            # 4 white glossy
    ((0, 0, 0), 0, (1, 1, 1), 0, 1, 2.2, 0, (.02, 5.1, 5.7), 13, 0),   # 5 glass
    ((.15, .48, .09), 0, (1, 1, 1), 0, 0, 2.6, 0, (0, 0, 0), 0, 0),    # 6 green glossy
    ((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 1),            # 7 light
    ((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 15),           # 8 light
]
# (type, material, TRANS, ROTAT, SCALE)
SAMPLE_OBJECTS = [
    ("cube", 0, (0, 0, 0), (0, 0, 90), (.01, 10, 10)),
    ("cube", 0, (0, 5, -5), (0, 90, 0), (.01, 10, 10)),
    ("cube", 0, (0, 10, 0), (0, 0, 90), (.01, 10, 10)),
    ("cube", 1, (-5, 5, 0), (0, 0, 0), (.01, 10, 10)),
    ("cube", 2, (5, 5, 0), (0, 0, 0), (.01, 10, 10)),
    ("sphere", 4, (0, 2, 0), (0, 180, 0), (3, 3, 3)),
    ("sphere", 3, (2, 5, 2), (0, 180, 0), (2.5, 2.5, 2.5)),
    ("sphere", 6, (-2, 5, -2), (0, 180, 0), (3, 3, 3)),
    ("cube", 8, (0, 10, 0), (0, 0, 90), (.3, 3, 3)),
]
SAMPLE_CAMERA = dict(res=(800, 800), fovy=25, iterations=5000, file="test.bmp",
                     frames=[((0, 4.5, 12), (0, 0, -1), (0, 1, 0))])


def _n(v):
    return repr(float(v)) if float(v) != int(v) else str(int(v))


def _v(t):
    return " ".join(_n(x) for x in t)


def scene_text(materials, camera, objects, lens=None):
    out = []
    for i, (rgb, specex, specrgb, refl, refr, ior, scatter, absc, rsct, emit) in enumerate(materials):
        out += ["MATERIAL %d" % i, "RGB         " + _v(rgb), "SPECEX      " + _n(specex), "SPECRGB     " + _v(specrgb),
                "REFL        " + _n(refl), "REFR        " + _n(refr), "REFRIOR     " + _n(ior),
                "SCATTER     " + _n(scatter), "ABSCOEFF    " + _v(absc), "RSCTCOEFF   " + _n(rsct),
                "EMITTANCE   " + _n(emit), ""]
    out += ["CAMERA", "RES         %d %d" % camera["res"], "FOVY        " + _n(camera["fovy"]),
            "ITERATIONS  %d" % camera["iterations"], "FILE        " + camera["file"]]
    for k, (eye, view, up) in enumerate(camera["frames"]):
        out += ["frame %d" % k, "EYE         " + _v(eye), "VIEW        " + _v(view), "UP          " + _v(up)]
    out.append("")
    if lens is not None:
        # top-level block the reference's dispatcher ignores (src/scene.cpp:22-31)
        out += ["LENS", "APERTURE    " + _n(lens[0]), "FOCALDIST   " + _n(lens[1]), ""]
    for i, (typ, mat, frames) in enumerate(objects):
        out += ["OBJECT %d" % i, typ, "material %d" % mat]
        for k, (t, r, s) in enumerate(frames):
            out += ["frame %d" % k, "TRANS       " + _v(t), "ROTAT       " + _v(r), "SCALE       " + _v(s)]
        out.append("")
    return "\n".join(out[:-1])  # like the shipped file: no trailing newline after the last object


def sample_scene(res=(800, 800), iterations=5000):
    cam = dict(SAMPLE_CAMERA, res=res, iterations=iterations)
    objs = [(t, m, [(tr, ro, sc)]) for (t, m, tr, ro, sc) in SAMPLE_OBJECTS]
    return scene_text(SAMPLE_MATERIALS, cam, objs)


def cornell_glass_dof():
    mats = [
        ((.85, .85, .85), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),   # 0 white
        ((.63, .06, .04), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),   # 1 red
        ((.15, .48, .09), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),   # 2 green
        ((1, 1, 1), 0, (1, 1, 1), 0, 1, 1.5, 0, (0, 0, 0), 0, 0),        # 3 clear glass
        ((.9, .95, 1), 0, (1, 1, 1), 0, 1, 1.33, 0, (0, 0, 0), 0, 0),    # 4 bluish glass
        ((1, 1, 1), 0, (.95, .95, .95), 1, 0, 0, 0, (0, 0, 0), 0, 0),    # 5 mirror
        ((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 15),         # 6 light
        ((.2, .3, .8), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),       # 7 blue diffuse
    ]
    z0 = (0, 0, 0)
    objs = [
        ("cube", 0, [((0, 0, 5), z0, (10, .01, 20))]),      # floor
        ("cube", 0, [((0, 10, 5), z0, (10, .01, 20))]),     # ceiling
        ("cube", 0, [((0, 5, -5), z0, (10, 10, .01))]),     # back
        ("cube", 0, [((0, 5, 15), z0, (10, 10, .01))]),     # front (behind the camera): closed box
        ("cube", 1, [((-5, 5, 5), z0, (.01, 10, 20))]),     # left
        ("cube", 2, [((5, 5, 5), z0, (.01, 10, 20))]),      # right
        ("cube", 6, [((0, 9.9, 1), z0, (3, .15, 3))]),      # emissive panel
        ("sphere", 3, [((-2.2, 1.5, 1), z0, (3, 3, 3))]),   # glass sphere
        ("sphere", 4, [((2.4, 1.25, 3.5), z0, (2.5, 2.5, 2.5))]),  # glass sphere, in front of the focal plane
        ("sphere", 5, [((1.2, 2, -2), z0, (4, 4, 4))]),     # mirror sphere
        ("cube", 3, [((-1, 1, 5), (0, .6, 0), (1.6, 2, 1.6))]),    # glass cube (rotated .6 rad about y)
        ("sphere", 7, [((-3.2, 4.5, -2.5), z0, (2, 2, 2))]),       # diffuse sphere
    ]
    cam = dict(res=(1920, 1080), fovy=22, iterations=4096, file="cornell.png",
               frames=[((0, 5, 14), (0, 0, -1), (0, 1, 0))])
    return scene_text(mats, cam, objs, lens=(0.12, 13.0))


def cornell_sss():
    mats = [
        ((.85, .85, .85), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 0 white
        ((.63, .06, .04), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 1 red
        ((.15, .48, .09), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 2 green
        ((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 15),             # 3 light
        ((1, 1, 1), 0, (1, 1, 1), 0, 1, 2.2, 1, (.02, 5.1, 5.7), 13, 0),     # 4 scattering medium
    ]
    z0 = (0, 0, 0)
    objs = [
        ("cube", 0, [((0, 0, 0), z0, (10, .01, 10))]),      # floor
        ("cube", 0, [((0, 10, 0), z0, (10, .01, 10))]),     # ceiling
        ("cube", 0, [((0, 5, -5), z0, (10, 10, .01))]),     # back
        ("cube", 0, [((0, 5, 5), z0, (10, 10, .01))]),      # front (behind the camera): closed room
        ("cube", 1, [((-5, 5, 0), z0, (.01, 10, 10))]),     # left
        ("cube", 2, [((5, 5, 0), z0, (.01, 10, 10))]),      # right
        ("cube", 3, [((0, 9.9, 0), z0, (3, .15, 3))]),      # emissive panel
        ("sphere", 4, [((-1.8, 1.6, -1), z0, (3.2, 3.2, 3.2))]),
        ("cube", 4, [((1.9, 1.25, 0.5), (0, .5, 0), (2.5, 2.5, 2.5))]),  # rotated .5 rad about y
    ]
    cam = dict(res=(800, 800), fovy=30, iterations=1024, file="cornell_sss.png",
               frames=[((0, 5, 4.8), (0, -0.25, -1), (0, 1, 0))])
    return scene_text(mats, cam, objs)


def cornell_glossy():
    mats = [
        ((.85, .85, .85), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 0 white
        ((.63, .06, .04), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 1 red
        ((.15, .48, .09), 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0),        # 2 green
        ((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 15),             # 3 light
        ((1, 1, 1), 10, (.95, .8, .5), 1, 0, 0, 0, (0, 0, 0), 0, 0),         # 4 glossy, SPECEX 10
        ((1, 1, 1), 100, (.9, .9, .9), 1, 0, 0, 0, (0, 0, 0), 0, 0),         # 5 glossy, SPECEX 100
        ((1, 1, 1), 1000, (.6, .75, .95), 1, 0, 0, 0, (0, 0, 0), 0, 0),      # 6 glossy, SPECEX 1000
        ((1, 1, 1), 0, (.95, .95, .95), 1, 0, 0, 0, (0, 0, 0), 0, 0),        # 7 perfect mirror
        ((1, 1, 1), 30, (.8, .8, .8), 1, 0, 0, 0, (0, 0, 0), 0, 0),          # 8 glossy wall, SPECEX 30
    ]
    z0 = (0, 0, 0)
    objs = [
        ("cube", 0, [((0, 0, 0), z0, (10, .01, 10))]),      # floor
        ("cube", 0, [((0, 10, 0), z0, (10, .01, 10))]),     # ceiling
        ("cube", 8, [((0, 5, -5), z0, (10, 10, .01))]),     # back: glossy
        ("cube", 0, [((0, 5, 5), z0, (10, 10, .01))]),      # front (behind the camera): closed room
        ("cube", 1, [((-5, 5, 0), z0, (.01, 10, 10))]),     # left
        ("cube", 2, [((5, 5, 0), z0, (.01, 10, 10))]),      # right
        ("cube", 3, [((0, 9.9, 0), z0, (3, .15, 3))]),      # emissive panel
        ("sphere", 4, [((-3, 1, -1.5), z0, (2, 2, 2))]),
        ("sphere", 5, [((-1, 1, -1.5), z0, (2, 2, 2))]),
        ("sphere", 6, [((1, 1, -1.5), z0, (2, 2, 2))]),
        ("sphere", 7, [((3, 1, -1.5), z0, (2, 2, 2))]),     # mirror
    ]
    cam = dict(res=(800, 800), fovy=30, iterations=1024, file="cornell_glossy.png",
               frames=[((0, 5, 4.8), (0, -0.25, -1), (0, 1, 0))])
    return scene_text(mats, cam, objs)


def sample_animated(n_frames=3, res=(800, 800), iterations=5000):
    """the sample scene with a bouncing sphere, a sliding camera and one per-frame array for every object
    (the reference's loader reads `frame k` blocks into per-frame arrays, src/scene.cpp:82-128, and its main loop
    advances through them, src/main.cpp:147-157)"""
    objs = []
    for i, (t, m, tr, ro, sc) in enumerate(SAMPLE_OBJECTS):
        frames = []
        for k in range(n_frames):
            tk = tr if i != 5 else (tr[0] + 0.5 * k, tr[1] + 1.2 * k, tr[2])   # object 5: the big sphere moves
            frames.append((tk, ro, sc))
        objs.append((t, m, frames))
    cam = dict(SAMPLE_CAMERA, res=res, iterations=iterations,
               frames=[((0.4 * k, 4.5, 12), (-0.03 * k, 0, -1), (0, 1, 0)) for k in range(n_frames)])
    return scene_text(SAMPLE_MATERIALS, cam, objs)


def procedural(n, seed=565, res=(1920, 1080), iterations=1024):
    rng = np.random.default_rng(seed)
    colours = [(.8, .8, .8), (.63, .06, .04), (.15, .48, .09), (.2, .3, .8), (.8, .7, .2), (.6, .2, .7)]
    mats = [(c, 0, (1, 1, 1), 0, 0, 0, 0, (0, 0, 0), 0, 0) for c in colours]
    mats.append(((1, 1, 1), 0, (.95, .95, .95), 1, 0, 0, 0, (0, 0, 0), 0, 0))  # 6 mirror
    mats.append(((1, 1, 1), 0, (1, 1, 1), 0, 1, 1.5, 0, (0, 0, 0), 0, 0))      # 7 glass
    mats.append(((1, 1, 1), 0, (0, 0, 0), 0, 0, 0, 0, (0, 0, 0), 0, 12))       # 8 light
    objs = [("cube", 0, [((0, -0.25, 0), (0, 0, 0), (40, .5, 40))])]           # ground slab
    for _ in range(n - 1):
        typ = "sphere" if rng.random() < 0.5 else "cube"
        u = rng.random()
        mat = 8 if u < 0.01 else 7 if u < 0.06 else 6 if u < 0.11 else int(rng.integers(0, 6))
        c = (round(float(rng.uniform(-12, 12)), 4), round(float(rng.uniform(0.2, 8)), 4), round(float(rng.uniform(-12, 12)), 4))
        s = round(float(rng.uniform(0.05, 0.3)), 4)
        r = tuple(round(float(x), 4) for x in rng.uniform(0, 6.2831, 3))
        objs.append((typ, mat, [(c, r, (s, s, s))]))
    cam = dict(res=res, iterations=iterations, fovy=25, file="procedural.png",
               frames=[((0, 6, 26), (0, -0.12, -1), (0, 1, 0))])
    return scene_text(mats, cam, objs)


def write_all():
    files = {"sample.txt": sample_scene(), "cornell_glass_dof.txt": cornell_glass_dof(),
             "sample_4k.txt": sample_scene((3840, 2160), 16384), "cornell_sss.txt": cornell_sss(),
             "cornell_glossy.txt": cornell_glossy()}
    for name, text in files.items():
        with open(os.path.join(HERE, name), "w") as f:
            f.write(text)
    return sorted(files)


if __name__ == "__main__":
    if len(sys.argv) >= 4 and sys.argv[1] == "--procedural":
        with open(sys.argv[3], "w") as f:
            f.write(procedural(int(sys.argv[2])))
    else:
        print(write_all())
