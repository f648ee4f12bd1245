"""The scene-file loader (pt_scene_load) against the reference loader's behaviour (src/scene.cpp)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scenes"))
import gen_scenes  # noqa: E402

from oracle_py import Ref  # noqa: E402


def test_sample_scene_parses_to_the_reference_structs_bitwise(pt, sample_scene):
    """scenes/sample.txt through OUR loader == the reference loader's parse of its own sampleScene.txt (golden)"""
    s = pt.Scene(os.path.join(ROOT, "scenes", "sample.txt"))
    assert (s.n_geoms, s.n_materials, s.n_frames) == (9, 9, 1)
    assert (s.width, s.height, s.iterations, s.image_name) == (800, 800, 5000, "test.bmp")
    g, m, cam, lens = s.frame(0)
    assert g.tobytes() == sample_scene["geoms"].tobytes(), "transforms must be bit-identical to glm's"
    assert m.tobytes() == sample_scene["materials"].tobytes()
    assert cam.tobytes() == sample_scene["camera"].tobytes()
    assert lens == (0.0, 0.0)
    # the ROTAT-is-radians quirk (SURVEY.md D1): cos(90 rad) = -0.448 shows up in object 0
    assert abs(g[0]["transform"][1] / 10 - (-np.sin(90.0))) < 1e-6


def test_generated_scene_files_are_current():
    for name, text in (("sample.txt", gen_scenes.sample_scene()), ("cornell_glass_dof.txt", gen_scenes.cornell_glass_dof()),
                       ("sample_4k.txt", gen_scenes.sample_scene((3840, 2160), 16384))):
        assert open(os.path.join(ROOT, "scenes", name)).read() == text, name


@pytest.mark.parametrize("eol", ["\n", "\r\n", "\r"])
def test_line_endings_and_missing_final_newline(pt, tmp_path, sample_scene, eol):
    """safeGetline accepts LF, CRLF, CR and a last line without terminator (src/utilities.cpp:109-139)"""
    text = gen_scenes.sample_scene().replace("\n", eol)
    for tail in ("", eol, eol + eol):
        p = tmp_path / "s.txt"
        p.write_bytes((text + tail).encode())
        g, m, cam, _ = pt.Scene(p).frame(0)
        assert g.tobytes() == sample_scene["geoms"].tobytes() and cam.tobytes() == sample_scene["camera"].tobytes()


def test_lens_block_comments_unknown_blocks_and_frames(pt, tmp_path):
    text = gen_scenes.scene_text(
        gen_scenes.SAMPLE_MATERIALS[:2],
        dict(res=(64, 32), fovy=30, iterations=7, file="out.png",
             frames=[((0, 1, 5), (0, 0, -1), (0, 1, 0)), ((1, 1, 5), (0, 0, -1), (0, 1, 0))]),
        [("sphere", 1, [((0, 0, 0), (0, 0, 0), (1, 1, 1)), ((0, 1, 0), (0, 0.5, 0), (1, 2, 1))]),
         ("cube", 0, [((0, -1, 0), (0, 0, 0), (4, .1, 4))]),
         ("bunny.obj", 0, [((0, 0, 0), (0, 0, 0), (1, 1, 1))])],
        lens=(0.25, 4.5))
    text = text.replace("MATERIAL 1", "MATERIAL 1   //a comment").replace("CAMERA", "SOMETHING new\nCAMERA", 1)
    p = tmp_path / "s.txt"
    p.write_text(text)
    s = pt.Scene(p)
    assert (s.n_geoms, s.n_materials, s.n_frames, s.width, s.height, s.iterations) == (3, 2, 2, 64, 32, 7)
    g0, m, cam0, lens = s.frame(0)
    g1, _, cam1, _ = s.frame(1)
    assert lens == (0.25, 4.5)
    assert g0[2]["type"] == pt.MESH and g0[0]["type"] == pt.SPHERE and g0[1]["type"] == pt.CUBE
    assert g1[0]["translation"].tolist() == [0, 1, 0] and g1[0]["scale"].tolist() == [1, 2, 1]
    assert g1[1].tobytes() == g0[1].tobytes()  # an object with one frame keeps it
    assert cam1["position"][0].tolist() == [1, 1, 5]
    # fov: half-angles in degrees, fovx from the aspect ratio (src/scene.cpp:203-207)
    assert cam0["fov"][0][1] == 30 and abs(np.tan(np.radians(cam0["fov"][0][0])) - 2 * np.tan(np.radians(30))) < 1e-5
    # inverse really is the inverse
    T = g1[0]["transform"].reshape(4, 4).astype(np.float64)
    assert np.allclose(T @ g1[0]["inverseTransform"].reshape(4, 4), np.eye(4), atol=1e-6)
    with pytest.raises(pt.PtError):
        s.frame(2)


def test_rotat_degrees_switch(pt, tmp_path):
    objs = [("cube", 0, [((0, 0, 0), (0, 0, 90), (1, 2, 3))])]
    cam = dict(res=(8, 8), fovy=25, iterations=1, file="a.png", frames=[((0, 0, 5), (0, 0, -1), (0, 1, 0))])
    p = tmp_path / "s.txt"
    p.write_text(gen_scenes.scene_text(gen_scenes.SAMPLE_MATERIALS[:1], cam, objs))
    rad = pt.Scene(p).frame(0)[0][0]["transform"].reshape(4, 4)
    deg = pt.Scene(p, rotat_degrees=True).frame(0)[0][0]["transform"].reshape(4, 4)
    assert abs(rad[0, 0] - np.cos(90.0)) < 1e-6        # reference behaviour: 90 radians
    assert abs(deg[0, 0]) < 1e-6 and abs(deg[1, 0] - 1) < 1e-6  # 90 degrees


def test_malformed_scenes_are_reported(pt, tmp_path):
    good = gen_scenes.sample_scene()
    cases = {
        "missing file": None,
        "material id": good.replace("MATERIAL 3", "MATERIAL 7", 1),
        "object id": good.replace("OBJECT 4", "OBJECT 9", 1),
        "object type": good.replace("sphere", "sphere ", 1),  # exact compare (src/scene.cpp:50-55)
        "frame number": good.replace("OBJECT 2\ncube\nmaterial 0\nframe 0", "OBJECT 2\ncube\nmaterial 0\nframe 1", 1),
        "no camera": good.replace("CAMERA", "CAMERAX", 1),
    }
    for name, text in cases.items():
        p = tmp_path / "bad.txt"
        if text is None:
            p = tmp_path / "does_not_exist.txt"
        else:
            p.write_text(text)
        with pytest.raises(pt.PtError):
            pt.Scene(p)
        assert pt.lib().pt_last_error(), name


@pytest.mark.skipif(not Ref.available(), reason="needs oracle/_ref")
def test_other_scenes_match_the_reference_loader_bitwise(pt, tmp_path):
    """non-square frames, rotations, 300 random objects: our loader == the reference's scene.cpp on the same file"""
    ref = Ref()
    files = [os.path.join(ROOT, "scenes", "cornell_glass_dof.txt"), os.path.join(ROOT, "scenes", "sample_4k.txt")]
    p = tmp_path / "proc.txt"
    p.write_text(gen_scenes.procedural(300, seed=3))
    files.append(str(p))
    for f in files:
        want = ref.load_scene(f)
        s = pt.Scene(f)
        g, m, cam, _ = s.frame(0)
        assert g.tobytes() == want["geoms"].tobytes(), f
        assert m.tobytes() == want["materials"].tobytes(), f
        assert cam.tobytes() == want["camera"].tobytes(), f
        assert (s.width, s.height, s.iterations, s.image_name) == (want["width"], want["height"], want["iterations"], want["image_name"])
