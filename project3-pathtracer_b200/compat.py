"""Python mirror of the reference's entry point

    void cudaRaytraceCore(uchar4* pos, camera* renderCam, int frame, int iterations,
                          material* materials, int numberOfMaterials, geom* geoms, int numberOfGeoms)

(reference src/raytraceKernel.h:17, called from src/main.cpp:110) through the C++ symbol libpt_b200.so exports.
The ctypes structures below are byte images of the reference's `geom`, `camera` and `material`
(src/sceneStructs.h:21-30,50-74; sizes 56 / 96 / 64, SURVEY.md appendix B)."""
import ctypes as C

import numpy as np

from . import GEOM_DTYPE, MATERIAL_DTYPE, lib

MANGLED = "_Z16cudaRaytraceCoreP6uchar4P6cameraiiP8materialiP4geomi"


class Vec3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


class Geom(C.Structure):
    _fields_ = [("type", C.c_int), ("materialid", C.c_int), ("frames", C.c_int),
                ("translations", C.c_void_p), ("rotations", C.c_void_p), ("scales", C.c_void_p),
                ("transforms", C.c_void_p), ("inverseTransforms", C.c_void_p)]


class Camera(C.Structure):
    _fields_ = [("resolution", C.c_float * 2), ("positions", C.c_void_p), ("views", C.c_void_p), ("ups", C.c_void_p),
                ("frames", C.c_int), ("fov", C.c_float * 2), ("iterations", C.c_uint), ("image", C.c_void_p),
                ("rayList", C.c_void_p), ("imageName", C.c_byte * 32)]  # std::string: never touched by the callee


assert C.sizeof(Geom) == 56 and C.sizeof(Camera) == 96


class RefScene:
    """geom[] / material[] / camera in the reference's host layout, built from per-frame flattened arrays
    (what scene.cpp leaves in scene::objects / materials / renderCam)."""

    def __init__(self, frames, materials, iterations=1):
        """frames: list of (geoms GEOM_DTYPE[n], camera CAMERA_DTYPE[1]) -- one entry per animation frame"""
        nf, n = len(frames), frames[0][0].shape[0]
        self.materials = np.ascontiguousarray(materials, dtype=MATERIAL_DTYPE)
        self._keep = []
        self.geoms = (Geom * n)()
        for i in range(n):
            cols = {k: np.ascontiguousarray(np.stack([f[0][i][k] for f in frames]), dtype=np.float32)
                    for k in ("translation", "rotation", "scale", "transform", "inverseTransform")}
            self._keep.append(cols)
            g = self.geoms[i]
            g.type, g.materialid, g.frames = int(frames[0][0][i]["type"]), int(frames[0][0][i]["materialid"]), nf
            g.translations, g.rotations, g.scales = (cols[k].ctypes.data for k in ("translation", "rotation", "scale"))
            g.transforms, g.inverseTransforms = cols["transform"].ctypes.data, cols["inverseTransform"].ctypes.data
        cam0 = frames[0][1].reshape(-1)[0]
        self.W, self.H = int(cam0["resolution"][0]), int(cam0["resolution"][1])
        self._pos = np.ascontiguousarray(np.stack([f[1].reshape(-1)[0]["position"] for f in frames]), dtype=np.float32)
        self._view = np.ascontiguousarray(np.stack([f[1].reshape(-1)[0]["view"] for f in frames]), dtype=np.float32)
        self._up = np.ascontiguousarray(np.stack([f[1].reshape(-1)[0]["up"] for f in frames]), dtype=np.float32)
        self.image = np.zeros((self.W * self.H, 3), np.float32)  # renderCam->image, the running mean
        c = self.camera = Camera()
        c.resolution[0], c.resolution[1] = self.W, self.H
        c.positions, c.views, c.ups = self._pos.ctypes.data, self._view.ctypes.data, self._up.ctypes.data
        c.frames = nf
        c.fov[0], c.fov[1] = float(cam0["fov"][0]), float(cam0["fov"][1])
        c.iterations = iterations
        c.image = self.image.ctypes.data
        c.rayList = None


def cudaRaytraceCore(pos, renderCam, frame, iterations, materials, numberOfMaterials, geoms, numberOfGeoms):
    """Same arguments as the reference.  `pos`: device pointer (int) of W*H uchar4 or None; renderCam: Camera;
    materials: numpy MATERIAL_DTYPE array; geoms: ctypes array of Geom."""
    fn = getattr(lib(), MANGLED)
    fn.restype = None
    m = np.ascontiguousarray(materials, dtype=MATERIAL_DTYPE)
    fn(C.c_void_p(pos), C.byref(renderCam), C.c_int(frame), C.c_int(iterations), m.ctypes.data_as(C.c_void_p),
       C.c_int(numberOfMaterials), geoms, C.c_int(numberOfGeoms))


def set_trace_depth(depth):
    if lib().pt_compat_set_trace_depth(C.c_int(depth)) != 0:
        raise ValueError("depth outside [1,64]")


def set_seed(seed):
    lib().pt_compat_set_seed(C.c_ulonglong(seed))


def set_lens(aperture, focal_distance):
    lib().pt_compat_set_lens(C.c_float(aperture), C.c_float(focal_distance))


def set_ahead(samples):
    """samples per group traced ahead of the calls (pt_compat_set_ahead)"""
    if lib().pt_compat_set_ahead(C.c_int(samples)) != 0:
        raise ValueError("samples outside [1, 64]")


def set_exit_on_error(on):
    lib().pt_compat_set_exit_on_error(C.c_int(1 if on else 0))


def set_direct_lighting(on):
    lib().pt_compat_set_direct_lighting(C.c_int(1 if on else 0))


def set_subsurface(on):
    lib().pt_compat_set_subsurface(C.c_int(1 if on else 0))


def set_glossy(on):
    lib().pt_compat_set_glossy(C.c_int(1 if on else 0))


def set_reference_stub(on):
    lib().pt_compat_set_reference_stub(C.c_int(1 if on else 0))


def last_status():
    return int(lib().pt_compat_last_status())


def reset():
    lib().pt_compat_reset()
