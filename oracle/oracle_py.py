"""TEST INFRASTRUCTURE ONLY: ctypes bindings for oracle/libpt_oracle.so (the C restatement) and,
where it exists, oracle/_ref/libptref.so (the reference's own functions compiled for the host).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "libpt_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libptref.so")
REF_GPU_SO = os.path.join(HERE, "_ref", "libptref_gpu.so")  # the reference's own (stub) kernels for sm_100a


class RefGpu:
    """The reference's own cudaRaytraceCore and kernels (oracle/ref_kernel_shim.cu); needs a GPU except noise_host."""

    @staticmethod
    def available():
        return os.path.exists(REF_GPU_SO)

    def __init__(self):
        self.lib = C.CDLL(REF_GPU_SO)

    def noise_host(self, W, H, time):
        out = np.zeros((W * H, 3), np.float32)
        self.lib.ref_noise_host(C.c_int(W), C.c_int(H), C.c_float(time), out.ctypes.data_as(C.c_void_p))
        return out

    def cudaRaytraceCore(self, W, H, iterations, image=None):
        """one call of the reference's entry point: returns (renderCam->image afterwards, the PBO bytes)"""
        img = np.zeros((W * H, 3), np.float32) if image is None else np.ascontiguousarray(image, np.float32).copy()
        pbo = np.zeros((W * H, 4), np.uint8)
        rc = self.lib.ref_cudaRaytraceCore(C.c_int(W), C.c_int(H), C.c_int(iterations), img.ctypes.data_as(C.c_void_p),
                                           pbo.ctypes.data_as(C.c_void_p))
        if rc != 0:
            raise RuntimeError("ref_cudaRaytraceCore: CUDA error %d" % rc)
        return img, pbo

GEOM_DTYPE = np.dtype(
    [
        ("type", "<i4"),
        ("materialid", "<i4"),
        ("translation", "<f4", (3,)),
        ("rotation", "<f4", (3,)),
        ("scale", "<f4", (3,)),
        ("transform", "<f4", (16,)),
        ("inverseTransform", "<f4", (16,)),
    ]
)
MATERIAL_DTYPE = np.dtype(
    [
        ("color", "<f4", (3,)),
        ("specularExponent", "<f4"),
        ("specularColor", "<f4", (3,)),
        ("hasReflective", "<f4"),
        ("hasRefractive", "<f4"),
        ("indexOfRefraction", "<f4"),
        ("hasScatter", "<f4"),
        ("absorptionCoefficient", "<f4", (3,)),
        ("reducedScatterCoefficient", "<f4"),
        ("emittance", "<f4"),
    ]
)
CAMERA_DTYPE = np.dtype(
    [
        ("resolution", "<f4", (2,)),
        ("position", "<f4", (3,)),
        ("view", "<f4", (3,)),
        ("up", "<f4", (3,)),
        ("fov", "<f4", (2,)),
    ]
)
assert GEOM_DTYPE.itemsize == 172 and MATERIAL_DTYPE.itemsize == 64 and CAMERA_DTYPE.itemsize == 52


class OrLens(C.Structure):
    _fields_ = [("aperture", C.c_float), ("focal_distance", C.c_float)]


class OrCamera(C.Structure):
    _fields_ = [
        ("resolution", C.c_float * 2),
        ("position", C.c_float * 3),
        ("view", C.c_float * 3),
        ("up", C.c_float * 3),
        ("fov", C.c_float * 2),
    ]


class OrScene(C.Structure):
    _fields_ = [
        ("geoms", C.c_void_p),
        ("n_geoms", C.c_int),
        ("materials", C.c_void_p),
        ("n_materials", C.c_int),
        ("cam", OrCamera),
        ("lens", OrLens),
        ("direct_lighting", C.c_int),
    ]


# a checkout of CIS565-Fall-2014/Project3-Pathtracer; oracle/_ref is built from it wherever it is present
REF_DIR = os.environ.get("PT_REFERENCE_DIR") or "/root/reference"


def build_oracle(force=False):
    """Compile the C restatement (and oracle/_ref when the reference checkout REF_DIR is present)."""
    if force or not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(
        os.path.join(HERE, "pt_oracle.c")
    ):
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])
    if os.path.isdir(os.path.join(REF_DIR, "src")):
        srcs = [os.path.join(HERE, "ref_shim.cu"), os.path.join(HERE, "ref_scene_shim.cpp"), os.path.join(HERE, "ref_kernel_shim.cu")]
        if force or not os.path.exists(REF_SO) or os.path.getmtime(REF_SO) < max(os.path.getmtime(s) for s in srcs):
            subprocess.check_call(["make", "-s", "-C", HERE, "ref", "REF=" + REF_DIR])
        # the drop-in build test: a host compiled against the reference's own headers, linked with libpt_b200.so
        dropin, main = os.path.join(HERE, "_ref", "ref_dropin"), os.path.join(HERE, "ref_dropin_main.cpp")
        lib = os.path.join(os.path.dirname(HERE), "project3-pathtracer_b200", "libpt_b200.so")
        if os.path.exists(lib) and (force or not os.path.exists(dropin) or os.path.getmtime(dropin) < os.path.getmtime(main)):
            subprocess.check_call(["make", "-s", "-C", HERE, "dropin", "REF=" + REF_DIR])


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    """The C restatement (oracle/pt_oracle.c)."""

    def __init__(self):
        build_oracle()
        L = self.lib = C.CDLL(ORACLE_SO)
        L.or_hash.restype = C.c_uint
        L.or_hash.argtypes = [C.c_uint]
        L.or_sphereIntersectionTest.restype = C.c_float
        L.or_boxIntersectionTest.restype = C.c_float
        L.or_u01.restype = C.c_float
        L.or_u01.argtypes = [C.c_uint32]
        L.or_render.restype = C.c_double
        L.or_render.argtypes = [
            C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32,
            C.c_void_p, C.c_void_p, C.c_int,
        ]
        L.or_render_ex.restype = C.c_double
        L.or_render_ex.argtypes = L.or_render.argtypes + [C.c_void_p]
        L.or_max_threads.restype = C.c_int
        L.or_refract.restype = C.c_int

    def hash(self, a):
        return int(self.lib.or_hash(C.c_uint(a & 0xFFFFFFFF)))

    def epsilonCheck(self, a, b):
        return bool(self.lib.or_epsilonCheck(C.c_float(a), C.c_float(b)))

    def ray_helpers(self, d):
        """(getInverseDirectionOfRay, getSignOfRay) of a direction"""
        d, inv, sign = _f32(d), np.zeros(3, np.float32), np.zeros(3, np.float32)
        self.lib.or_ray_helpers(_p(d), _p(inv), _p(sign))
        return inv, sign

    def multiplyMV(self, m16, v4):
        m, v, out = _f32(m16), _f32(v4), np.zeros(3, np.float32)
        self.lib.or_multiplyMV(_p(m), _p(v), _p(out))
        return out

    def getPointOnRay(self, o, d, t):
        o, d, out = _f32(o), _f32(d), np.zeros(3, np.float32)
        self.lib.or_getPointOnRay(_p(o), _p(d), C.c_float(t), _p(out))
        return out

    def getRadiuses(self, geom):
        g = np.ascontiguousarray(geom)
        out = np.zeros(3, np.float32)
        self.lib.or_getRadiuses(_p(g), _p(out))
        return out

    def noise_image(self, W, H, time, reversed_order):
        """generateRandomNumberFromThread over a W x H frame (the reference's stub renderer)"""
        out = np.zeros((W * H, 3), np.float32)
        self.lib.or_noise_image(C.c_int(W), C.c_int(H), C.c_float(time), C.c_int(1 if reversed_order else 0), _p(out))
        return out

    def random_points(self, geom, seeds):
        """getRandomPointOnCube / getRandomPointOnSphere (by geom type) for every float seed"""
        g, sd = np.ascontiguousarray(geom), _f32(seeds).ravel()
        out = np.zeros((sd.size, 3), np.float32)
        self.lib.or_random_points_batch(_p(g), C.c_int(sd.size), _p(sd), _p(out))
        return out

    def points_u(self, geom, u):
        """the same samplers driven by given uniforms, u = (n, 3)"""
        g, u = np.ascontiguousarray(geom), _f32(u).reshape(-1, 3)
        out = np.zeros_like(u)
        self.lib.or_points_u_batch(_p(g), C.c_int(u.shape[0]), _p(u), _p(out))
        return out

    def sphere_dirs(self, xi1, xi2):
        xi1, xi2 = _f32(xi1).ravel(), _f32(xi2).ravel()
        out = np.zeros((xi1.size, 3), np.float32)
        self.lib.or_sphere_dirs_batch(C.c_int(xi1.size), _p(xi1), _p(xi2), _p(out))
        return out

    def transmission(self, absorption, distance):
        a, d = _f32(absorption).reshape(-1, 3), _f32(distance).ravel()
        out = np.zeros_like(a)
        self.lib.or_transmission_batch(C.c_int(d.size), _p(a), _p(d), _p(out))
        return out

    def intersect_one(self, geom, which, o, d):
        """rays (n,3) against one geom with the sphere (0) or box (1) test."""
        g = np.ascontiguousarray(geom)
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        t, p, nr = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        fn = self.lib.or_sphereIntersectionTest if which == 0 else self.lib.or_boxIntersectionTest
        for i in range(n):
            t[i] = fn(_p(g), _p(o[i]), _p(d[i]), _p(p[i]), _p(nr[i]))
        return t, p, nr

    def hemisphere(self, normal, xi1, xi2, ref=False):
        normal = _f32(normal).reshape(-1, 3)
        xi1, xi2 = _f32(xi1).ravel(), _f32(xi2).ravel()
        out = np.zeros_like(normal)
        fn = self.lib.or_hemisphere_ref if ref else self.lib.or_hemisphere
        for i in range(normal.shape[0]):
            fn(_p(normal[i]), C.c_float(xi1[i]), C.c_float(xi2[i]), _p(out[i]))
        return out

    def philox(self, ctr, key):
        c = np.ascontiguousarray(ctr, dtype=np.uint32)
        k = np.ascontiguousarray(key, dtype=np.uint32)
        out = np.zeros(4, np.uint32)
        self.lib.or_philox4x32_10(_p(c), _p(k), _p(out))
        return out

    def u01(self, x):
        return float(self.lib.or_u01(C.c_uint32(x)))

    def sincos_2pi(self, u):
        s, c = C.c_float(), C.c_float()
        self.lib.or_sincos_2pi(C.c_float(u), C.byref(s), C.byref(c))
        return s.value, c.value

    def reflect(self, n, i):
        n, i, out = _f32(n), _f32(i), np.zeros(3, np.float32)
        self.lib.or_reflect(_p(n), _p(i), _p(out))
        return out

    def refract(self, n, i, ior_i, ior_t):
        n, i, out = _f32(n), _f32(i), np.zeros(3, np.float32)
        tir = self.lib.or_refract(_p(n), _p(i), C.c_float(ior_i), C.c_float(ior_t), _p(out))
        return int(tir), out

    def fresnel(self, n, i, ior_i, ior_t, trans, tir):
        n, i, tr = _f32(n), _f32(i), _f32(trans)
        R, T = C.c_float(), C.c_float()
        self.lib.or_fresnel(_p(n), _p(i), C.c_float(ior_i), C.c_float(ior_t), _p(n), _p(tr), C.c_int(tir),
                            C.byref(R), C.byref(T))
        return R.value, T.value

    @staticmethod
    def _cam(cam):
        c = OrCamera()
        a = np.ascontiguousarray(cam).view(np.float32).ravel()
        C.memmove(C.byref(c), a.ctypes.data, 52)
        return c

    def raygen(self, cam, lens, seed, pixel, sample):
        c = self._cam(cam)
        l = OrLens(float(lens[0]), float(lens[1]))
        pixel = np.ascontiguousarray(pixel, dtype=np.uint32).ravel()
        sample = np.ascontiguousarray(sample, dtype=np.uint32).ravel()
        n = pixel.shape[0]
        o, d = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        self.lib.or_raygen_batch(C.byref(c), C.byref(l), C.c_uint64(seed), C.c_int(n), _p(pixel), _p(sample), _p(o), _p(d))
        return o, d

    def intersect_rays(self, geoms, o, d):
        g = np.ascontiguousarray(geoms)
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        gid, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
        p, nr = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        self.lib.or_intersect_rays(_p(g), C.c_int(g.shape[0]), C.c_int(n), _p(o), _p(d), _p(gid), _p(t), _p(p), _p(nr))
        return gid, t, p, nr

    def make_scene(self, geoms, materials, cam, lens=(0.0, 0.0), direct_lighting=False):
        g = np.ascontiguousarray(geoms)
        m = np.ascontiguousarray(materials)
        sc = OrScene()
        sc.geoms, sc.n_geoms = g.ctypes.data, g.shape[0]
        sc.materials, sc.n_materials = m.ctypes.data, m.shape[0]
        sc.cam = self._cam(cam)
        sc.lens = OrLens(float(lens[0]), float(lens[1]))
        sc.direct_lighting = 1 if direct_lighting else 0
        sc._keep = (g, m)
        return sc

    def render(self, scene, first_sample, n_samples, max_depth, seed, pix_begin=0, pix_end=None, threads=0,
               sum_rgb=None):
        W, H = int(scene.cam.resolution[0]), int(scene.cam.resolution[1])
        if pix_end is None:
            pix_end = W * H
        if sum_rgb is None:
            sum_rgb = np.zeros((W * H, 3), np.float32)
        live = np.zeros(64, np.uint64)
        shadow = C.c_uint64(0)
        secs = self.lib.or_render_ex(C.byref(scene), first_sample, n_samples, max_depth, seed, pix_begin, pix_end,
                                     _p(sum_rgb), _p(live), threads, C.byref(shadow))
        self.last_shadow_rays = int(shadow.value)
        return sum_rgb, live[:max_depth].copy(), float(secs)

    def max_threads(self):
        return int(self.lib.or_max_threads())


class Ref:
    """The reference's own functions (oracle/_ref/libptref.so).  Exists only where it was built."""

    @staticmethod
    def available():
        return os.path.exists(REF_SO)

    def __init__(self):
        L = self.lib = C.CDLL(REF_SO)
        L.ref_hash.restype = C.c_uint
        L.ref_hash.argtypes = [C.c_uint]
        L.refscene_load.restype = C.c_void_p
        L.refscene_load.argtypes = [C.c_char_p]

    def hash(self, a):
        return int(self.lib.ref_hash(C.c_uint(a & 0xFFFFFFFF)))

    def multiplyMV(self, m16, v4):
        m, v, out = _f32(m16), _f32(v4), np.zeros(3, np.float32)
        self.lib.ref_multiplyMV(_p(m), _p(v), _p(out))
        return out

    def getPointOnRay(self, o, d, t):
        o, d, out = _f32(o), _f32(d), np.zeros(3, np.float32)
        self.lib.ref_getPointOnRay(_p(o), _p(d), C.c_float(t), _p(out))
        return out

    def getRadiuses(self, geom):
        g = np.ascontiguousarray(geom)
        out = np.zeros(3, np.float32)
        self.lib.ref_getRadiuses(_p(g), _p(out))
        return out

    def intersect_one(self, geom, which, o, d):
        g = np.ascontiguousarray(geom)
        o, d = _f32(o).reshape(-1, 3), _f32(d).reshape(-1, 3)
        n = o.shape[0]
        t, p, nr = np.zeros(n, np.float32), np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        self.lib.ref_intersect_batch(_p(g), C.c_int(which), C.c_int(n), _p(o), _p(d), _p(t), _p(p), _p(nr))
        return t, p, nr

    def hemisphere(self, normal, xi1, xi2):
        normal = _f32(normal).reshape(-1, 3)
        xi1, xi2 = _f32(xi1).ravel(), _f32(xi2).ravel()
        out = np.zeros_like(normal)
        self.lib.ref_hemisphere_batch(C.c_int(normal.shape[0]), _p(normal), _p(xi1), _p(xi2), _p(out))
        return out

    def epsilonCheck(self, a, b):
        return bool(self.lib.ref_epsilonCheck(C.c_float(a), C.c_float(b)))

    def ray_helpers(self, d):
        d, inv, sign = _f32(d), np.zeros(3, np.float32), np.zeros(3, np.float32)
        self.lib.ref_ray_helpers(_p(d), _p(inv), _p(sign))
        return inv, sign

    def random_points_on_cube(self, geom, seeds):
        g, sd = np.ascontiguousarray(geom), _f32(seeds).ravel()
        out = np.zeros((sd.size, 3), np.float32)
        self.lib.ref_getRandomPointOnCube_batch(_p(g), C.c_int(sd.size), _p(sd), _p(out))
        return out

    def sampling_stubs(self):
        out = np.zeros(9, np.float32)
        self.lib.ref_sampling_stubs(_p(out))
        return out

    def bsdf_stub(self):
        return int(self.lib.ref_calculateBSDF_stub())

    def layout(self):
        out = (C.c_int * 64)()
        n = self.lib.ref_layout(out, 64)
        return [int(out[i]) for i in range(n)]

    def load_scene(self, path, frame=0):
        h = self.lib.refscene_load(path.encode())
        ng, nm, fr, it, w, hh = (C.c_int() for _ in range(6))
        self.lib.refscene_counts(C.c_void_p(h), *(C.byref(x) for x in (ng, nm, fr, it, w, hh)))
        geoms = np.zeros(ng.value, GEOM_DTYPE)
        mats = np.zeros(nm.value, MATERIAL_DTYPE)
        cam = np.zeros(1, CAMERA_DTYPE)
        name = C.create_string_buffer(256)
        self.lib.refscene_static_geoms(C.c_void_p(h), C.c_int(frame), _p(geoms))
        self.lib.refscene_materials(C.c_void_p(h), _p(mats))
        self.lib.refscene_camera(C.c_void_p(h), C.c_int(frame), _p(cam), name, 256)
        return dict(geoms=geoms, materials=mats, camera=cam, frames=fr.value, iterations=it.value,
                    width=w.value, height=hh.value, image_name=name.value.decode())

    def save_image(self, rgb, W, H, image_name, frame):
        rgb = _f32(rgb)
        out = C.create_string_buffer(512)
        self.lib.ref_save_image(_p(rgb), C.c_int(W), C.c_int(H), image_name.encode(), C.c_int(frame), out, 512)
        return out.value.decode()
