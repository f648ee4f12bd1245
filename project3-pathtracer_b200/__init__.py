"""project3-pathtracer_b200 -- host-side mirror of the reference interface over libpt_b200.so.

B200-native wavefront path tracer, drop-in for the hot path of CIS565-Fall-2014/Project3-Pathtracer
(cudaRaytraceCore, reference src/raytraceKernel.cu:108-165).  Everything here is a thin ctypes layer over the C ABI
declared in include/pt_b200.h; the compute lives in csrc/ (hand-written CUDA for sm_100a).

There is NO CPU fallback: if the shared library is missing or no CUDA device is present, calls raise.

The directory name contains a hyphen, so import it with importlib:

    import importlib; pt = importlib.import_module("project3-pathtracer_b200")
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libpt_b200.so")

# numpy images of the reference structs (src/sceneStructs.h:32-48,63-74)
GEOM_DTYPE = np.dtype([("type", "<i4"), ("materialid", "<i4"), ("translation", "<f4", (3,)), ("rotation", "<f4", (3,)),
                       ("scale", "<f4", (3,)), ("transform", "<f4", (16,)), ("inverseTransform", "<f4", (16,))])
MATERIAL_DTYPE = np.dtype([("color", "<f4", (3,)), ("specularExponent", "<f4"), ("specularColor", "<f4", (3,)),
                           ("hasReflective", "<f4"), ("hasRefractive", "<f4"), ("indexOfRefraction", "<f4"),
                           ("hasScatter", "<f4"), ("absorptionCoefficient", "<f4", (3,)),
                           ("reducedScatterCoefficient", "<f4"), ("emittance", "<f4")])
CAMERA_DTYPE = np.dtype([("resolution", "<f4", (2,)), ("position", "<f4", (3,)), ("view", "<f4", (3,)),
                         ("up", "<f4", (3,)), ("fov", "<f4", (2,))])
LENS_DTYPE = np.dtype([("aperture", "<f4"), ("focal_distance", "<f4")])
assert GEOM_DTYPE.itemsize == 172 and MATERIAL_DTYPE.itemsize == 64 and CAMERA_DTYPE.itemsize == 52

SPHERE, CUBE, MESH = 0, 1, 2
HIT_FILTERED, HIT_EXACT_SCAN = 0, 1  # pt_intersect_ex modes


class PtError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libpt_b200.so (building it first if sources are newer).  Fails loudly; never falls back."""
    global _lib
    if _lib is None:
        path = os.environ.get("PT_B200_LIB")  # developer knob: load an alternative build of the same library
        if not path:
            _build.build()
            path = LIB_PATH
        if not os.path.exists(path):
            raise PtError("%s is missing: the CUDA extension is required (no CPU fallback)" % path)
        _lib = C.CDLL(path)
        _lib.pt_last_error.restype = C.c_char_p
    return _lib


def _check(rc):
    if rc != 0:
        raise PtError("pt_b200 error %d: %s" % (rc, lib().pt_last_error().decode(errors="replace")))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _arr(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def device_count():
    n = C.c_int()
    _check(lib().pt_device_count(C.byref(n)))
    return n.value


class Context:
    """Scene + path-state buffers + accumulation image resident on one GPU (pt_context_* in include/pt_b200.h)."""

    def __init__(self, geoms, materials, camera, lens=None, device=0):
        self._h = C.c_void_p()
        g = _arr(geoms, GEOM_DTYPE)
        m = _arr(materials, MATERIAL_DTYPE)
        cam = _arr(camera, CAMERA_DTYPE).reshape(-1)[:1]
        ln = None if lens is None else np.array([(lens[0], lens[1])], LENS_DTYPE)
        _check(lib().pt_context_create(_p(g), C.c_int(g.shape[0]), _p(m), C.c_int(m.shape[0]), _p(cam),
                                       _p(ln) if ln is not None else None, C.c_int(device), C.byref(self._h)))
        self.width, self.height = int(cam["resolution"][0][0]), int(cam["resolution"][0][1])
        self.npix = self.width * self.height
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().pt_context_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def update_scene(self, geoms, materials, camera, lens=None):
        g, m = _arr(geoms, GEOM_DTYPE), _arr(materials, MATERIAL_DTYPE)
        cam = _arr(camera, CAMERA_DTYPE).reshape(-1)[:1]
        ln = None if lens is None else np.array([(lens[0], lens[1])], LENS_DTYPE)
        _check(lib().pt_update_scene(self._h, _p(g), C.c_int(g.shape[0]), _p(m), C.c_int(m.shape[0]), _p(cam),
                                     _p(ln) if ln is not None else None))

    def set_wavefront_paths(self, max_paths):
        _check(lib().pt_set_wavefront_paths(self._h, C.c_uint64(int(max_paths))))

    def set_stream(self, cuda_stream):
        _check(lib().pt_set_stream(self._h, C.c_void_p(cuda_stream)))

    def render(self, first_sample, n_samples, max_depth, seed=0):
        _check(lib().pt_render(self._h, C.c_uint32(first_sample), C.c_uint32(n_samples), C.c_int(max_depth),
                               C.c_uint64(seed)))

    def sync(self):
        _check(lib().pt_sync(self._h))

    def clear(self):
        _check(lib().pt_clear(self._h))

    def last_render_ms(self):
        ms = C.c_float()
        _check(lib().pt_last_render_ms(self._h, C.byref(ms)))
        return ms.value

    def download_sum(self, out=None):
        out = np.empty((self.npix, 3), np.float32) if out is None else out
        _check(lib().pt_download_sum(self._h, _p(out)))
        return out

    def download_mean(self, spp, out=None):
        out = np.empty((self.npix, 3), np.float32) if out is None else out
        _check(lib().pt_download_mean(self._h, _p(out), C.c_uint32(spp)))
        return out

    def stream_begin(self, first_sample, spp_before, max_depth, seed=0, group=8):
        """pt_stream_begin: trace samples first_sample, first_sample + 1, ... ahead, `group` at a time, on top of a sum
        of spp_before samples"""
        _check(lib().pt_stream_begin(self._h, C.c_uint32(first_sample), C.c_uint32(spp_before), C.c_int(max_depth),
                                     C.c_uint64(seed), C.c_uint32(group)))

    def stream_next(self, out=None, device_rgba8=None):
        """pt_stream_next: the running mean after the next traced sample -> (mean (W*H, 3), divisor)"""
        out = np.empty((self.npix, 3), np.float32) if out is None else out
        spp = C.c_uint32()
        _check(lib().pt_stream_next(self._h, _p(out), C.c_void_p(device_rgba8), C.byref(spp)))
        return out, spp.value

    def stream_end(self):
        _check(lib().pt_stream_end(self._h))

    def upload_sum(self, rgb):
        rgb = _arr(rgb, np.float32)
        assert rgb.size == self.npix * 3
        _check(lib().pt_upload_sum(self._h, _p(rgb)))

    def resolve_rgba8(self, spp, device_ptr=None):
        out = np.empty((self.npix, 4), np.uint8)
        _check(lib().pt_resolve_rgba8(self._h, C.c_uint32(spp), _p(out), C.c_void_p(device_ptr)))
        return out

    def accum_device_ptr(self):
        p, n = C.c_void_p(), C.c_size_t()
        _check(lib().pt_accum_device_ptr(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def counters(self):
        paths, segs = C.c_uint64(), C.c_uint64()
        live = np.zeros(64, np.uint64)
        _check(lib().pt_counters(self._h, C.byref(paths), C.byref(segs), _p(live)))
        return paths.value, segs.value, live

    def set_kernel_policy(self, bounce_kernel=0):
        """tuning / test knob (pt_set_kernel_policy): depths >= 1 of few-geom scenes run 0 = the kernel the scene's
        measured survival suggests, 1 = the re-batched kernel (k_bounce_q), 2 = the fused kernel; same results"""
        _check(lib().pt_set_kernel_policy(self._h, C.c_int(bounce_kernel)))

    def set_band_pixels(self, pixels):
        """pixels per wavefront band (0 = automatic); results do not depend on it"""
        _check(lib().pt_set_band_pixels(self._h, C.c_uint32(pixels)))

    def set_direct_lighting(self, on=True):
        """direct light sampling at diffuse bounces (pt_set_direct_lighting); off by default"""
        _check(lib().pt_set_direct_lighting(self._h, C.c_int(1 if on else 0)))

    def set_subsurface(self, on=True):
        """subsurface scattering inside refractive geoms whose material has SCATTER > 0 and RSCTCOEFF > 0
        (pt_set_subsurface); off by default"""
        _check(lib().pt_set_subsurface(self._h, C.c_int(1 if on else 0)))

    def set_glossy(self, on=True):
        """glossy reflection: reflective materials with SPECEX > 0 sample a Phong lobe around the mirror direction
        (pt_set_glossy); off by default"""
        _check(lib().pt_set_glossy(self._h, C.c_int(1 if on else 0)))

    def shadow_rays(self):
        """(shadow rays traced since the last clear, emissive geoms in the scene)"""
        n, nl = C.c_uint64(), C.c_int()
        _check(lib().pt_shadow_rays(self._h, C.byref(n), C.byref(nl)))
        return n.value, nl.value

    def launch_count(self):
        n = C.c_uint64()
        _check(lib().pt_launch_count(self._h, C.byref(n)))
        return n.value

    def raygen(self, seed, pixel, sample):
        pixel, sample = _arr(pixel, np.uint32).ravel(), _arr(sample, np.uint32).ravel()
        n = pixel.shape[0]
        o, d = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        _check(lib().pt_raygen(self._h, C.c_uint64(seed), C.c_int(n), _p(pixel), _p(sample), _p(o), _p(d)))
        return o, d

    def intersect(self, origin, direction, mode=HIT_FILTERED, with_stats=False):
        """closest hit of n rays -> (geom id, t, point, normal) [+ fallbacks]; mode HIT_EXACT_SCAN runs the exact test on
        every geom (the specification the filtered default must reproduce bit for bit)"""
        o, d = _arr(origin, np.float32).reshape(-1, 3), _arr(direction, np.float32).reshape(-1, 3)
        n = o.shape[0]
        gid, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
        p, nr = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        fb = C.c_uint64()
        _check(lib().pt_intersect_ex(self._h, C.c_int(mode), C.c_int(n), _p(o), _p(d), _p(gid), _p(t), _p(p), _p(nr),
                                     C.byref(fb)))
        return (gid, t, p, nr, fb.value) if with_stats else (gid, t, p, nr)

    def primary_hit(self, seed, pixel, sample, with_stats=False):
        """primary rays of (pixel, sample) pairs through depth 0's closest hit -- the per-pixel table's candidate first,
        then the filter -- -> (geom id, t, point, normal, decided) [+ fallbacks]; decided = the table settled the ray"""
        pixel, sample = _arr(pixel, np.uint32).ravel(), _arr(sample, np.uint32).ravel()
        n = pixel.shape[0]
        gid, t = np.zeros(n, np.int32), np.zeros(n, np.float32)
        p, nr = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        dec = np.zeros(n, np.uint8)
        fb = C.c_uint64()
        _check(lib().pt_primary_hit(self._h, C.c_uint64(seed), C.c_int(n), _p(pixel), _p(sample), _p(gid), _p(t), _p(p),
                                    _p(nr), _p(dec), C.byref(fb)))
        out = (gid, t, p, nr, dec.astype(bool))
        return out + (fb.value,) if with_stats else out

    def primary_table_info(self, time_build=False):
        """(the current scene and camera have the primary-ray table, ms of one rebuild or None)"""
        on, ms = C.c_int(), C.c_float()
        _check(lib().pt_primary_table_info(self._h, C.byref(on), C.byref(ms) if time_build else None))
        return bool(on.value), (ms.value if time_build else None)

    def set_filter_scale(self, scale):
        """test hook: multiply the rounding-error terms of the closest-hit filter's bounds (1 = shipped)"""
        _check(lib().pt_set_filter_scale(self._h, C.c_float(scale)))

    def filter_retries(self):
        """hierarchy scenes: segments since the last clear() that the second candidate's exact test settled (pt_filter_retries)"""
        n = C.c_uint64()
        _check(lib().pt_filter_retries(self._h, C.byref(n)))
        return n.value

    def filter_stats(self):
        """segments rendered since the last clear() whose closest hit fell back to the exact scan"""
        n = C.c_uint64()
        _check(lib().pt_filter_stats(self._h, C.byref(n)))
        return n.value


def reduce_to_first(contexts):
    """single-process multi-GPU combine: one ncclReduce(sum) of the accumulation images into contexts[0]"""
    arr = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    _check(lib().pt_reduce_to_first(arr, C.c_int(len(contexts))))


def selftest_math(device=0):
    """mismatches of the kernels' single-guard IEEE (sqrt, reciprocal, 1/sqrt) over all 2^32 inputs: must be (0, 0, 0)"""
    bad = (C.c_uint64 * 3)()
    _check(lib().pt_selftest_math(C.c_int(device), bad))
    return tuple(int(x) for x in bad)


def random_points_on_geom(geom, seeds, device=0):
    """getRandomPointOnCube / getRandomPointOnSphere (src/intersections.h:133-182), one world point per float seed"""
    g, sd = np.ascontiguousarray(geom), _arr(seeds, np.float32).ravel()
    out = np.zeros((sd.size, 3), np.float32)
    _check(lib().pt_random_points_on_geom(C.c_int(device), _p(g), C.c_int(sd.size), _p(sd), _p(out)))
    return out


def points_on_geom_u(geom, u, device=0):
    """the same samplers driven by given uniforms, u = (n, 3)"""
    g, u = np.ascontiguousarray(geom), _arr(u, np.float32).reshape(-1, 3)
    out = np.zeros_like(u)
    _check(lib().pt_points_on_geom_u(C.c_int(device), _p(g), C.c_int(u.shape[0]), _p(u), _p(out)))
    return out


def random_directions_in_sphere(xi1, xi2, device=0):
    """getRandomDirectionInSphere (src/interactions.h:93-95)"""
    a, b = _arr(xi1, np.float32).ravel(), _arr(xi2, np.float32).ravel()
    assert a.shape == b.shape
    out = np.zeros((a.size, 3), np.float32)
    _check(lib().pt_random_directions_in_sphere(C.c_int(device), C.c_int(a.size), _p(a), _p(b), _p(out)))
    return out


def calculate_transmission(absorption, distance, device=0):
    """calculateTransmission (src/interactions.h:31-33): exp(-absorption * distance) per channel"""
    a, d = _arr(absorption, np.float32).reshape(-1, 3), _arr(distance, np.float32).ravel()
    assert a.shape[0] == d.size
    out = np.zeros_like(a)
    _check(lib().pt_calculate_transmission(C.c_int(device), C.c_int(d.size), _p(a), _p(d), _p(out)))
    return out


def sample_medium(absorption, scatter, distance, u, device=0):
    """calculateScatterAndAbsorption (src/interactions.h:36-39), the free flight of subsurface scattering:
    u = (n, 3) uniforms (xi1, xi2, xf) -> (scattered bool (n,), s (n,), direction (n, 3), weight (n, 3)).
    s = -log(1 - xf) / scatter; where s < distance the segment scatters there into a uniform direction with weight
    exp(-absorption * s), elsewhere it passes with direction 0 and weight exp(-absorption * distance)."""
    a, sc = _arr(absorption, np.float32).reshape(-1, 3), _arr(scatter, np.float32).ravel()
    d, uu = _arr(distance, np.float32).ravel(), _arr(u, np.float32).reshape(-1, 3)
    n = d.size
    assert a.shape[0] == n and sc.size == n and uu.shape[0] == n
    flag, s = np.zeros(n, np.int32), np.zeros(n, np.float32)
    dirs, w = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
    _check(lib().pt_sample_medium(C.c_int(device), C.c_int(n), _p(a), _p(sc), _p(d), _p(uu), _p(flag), _p(s), _p(dirs), _p(w)))
    return flag.astype(bool), s, dirs, w


def sample_glossy(normal, incident, exponent, u, device=0):
    """the glossy lobe of pt_set_glossy: outward normal (n, 3), incident direction (n, 3), SPECEX (n,) and uniforms
    u = (n, 2) -> direction (n, 3), a Phong lobe of exponent SPECEX around the mirror direction of the normal turned to
    face the incident ray, folded above the surface"""
    nn, d = _arr(normal, np.float32).reshape(-1, 3), _arr(incident, np.float32).reshape(-1, 3)
    e, uu = _arr(exponent, np.float32).ravel(), _arr(u, np.float32).reshape(-1, 2)
    n = e.size
    assert nn.shape[0] == n and d.shape[0] == n and uu.shape[0] == n
    out = np.zeros((n, 3), np.float32)
    _check(lib().pt_sample_glossy(C.c_int(device), C.c_int(n), _p(nn), _p(d), _p(e), _p(uu), _p(out)))
    return out


STUB_ORDER_DEVICE, STUB_ORDER_HOST = 0, 1


def reference_stub_image(width, height, iterations, order=STUB_ORDER_DEVICE, device=0):
    """the noise image the reference's raytraceRay stub writes for this iteration (src/raytraceKernel.cu:93-104)"""
    out = np.zeros((width * height, 3), np.float32)
    _check(lib().pt_reference_stub_image(C.c_int(device), C.c_int(width), C.c_int(height), C.c_int(iterations),
                                         C.c_int(order), _p(out)))
    return out


def set_compact_mode(mode):
    """0 = count / scan / scatter (default), 1 = single pass with the look-back inside"""
    _check(lib().pt_set_compact_mode(C.c_int(mode)))


def compact_u32(values, flags, device=0):
    """Stream compaction primitive on its own (pt_compact_u32): values[flags != 0], order preserved."""
    v, f = _arr(values, np.uint32).ravel(), _arr(flags, np.uint8).ravel()
    assert v.shape == f.shape
    out = np.empty(max(v.shape[0], 1), np.uint32)
    n_out = C.c_uint64()
    _check(lib().pt_compact_u32(C.c_int(device), _p(v), _p(f), C.c_uint64(v.shape[0]), _p(out), C.byref(n_out)))
    return out[: n_out.value].copy()


def compact_u32_timed(values, flags, iters=10, device=0):
    """pt_compact_u32_timed: (compacted values, kernel milliseconds per launch on the device)"""
    v, f = _arr(values, np.uint32).ravel(), _arr(flags, np.uint8).ravel()
    assert v.shape == f.shape
    out = np.empty(max(v.shape[0], 1), np.uint32)
    n_out, ms = C.c_uint64(), C.c_float()
    _check(lib().pt_compact_u32_timed(C.c_int(device), _p(v), _p(f), C.c_uint64(v.shape[0]), _p(out), C.byref(n_out),
                                      C.c_int(iters), C.byref(ms)))
    return out[: n_out.value].copy(), ms.value


class Scene:
    """scene::scene(string) of the reference (src/scene.cpp:11-35) through pt_scene_load."""

    def __init__(self, path, rotat_degrees=False):
        self._h = C.c_void_p()
        _check(lib().pt_scene_load(str(path).encode(), C.c_int(1 if rotat_degrees else 0), C.byref(self._h)))
        ng, nm, nf, w, h, it = (C.c_int() for _ in range(6))
        name = C.create_string_buffer(512)
        _check(lib().pt_scene_info(self._h, C.byref(ng), C.byref(nm), C.byref(nf), C.byref(w), C.byref(h), C.byref(it),
                                   name, C.c_int(512)))
        self.n_geoms, self.n_materials, self.n_frames = ng.value, nm.value, nf.value
        self.width, self.height, self.iterations = w.value, h.value, it.value
        self.image_name = name.value.decode()

    def frame(self, frame=0):
        g = np.zeros(self.n_geoms, GEOM_DTYPE)
        m = np.zeros(self.n_materials, MATERIAL_DTYPE)
        cam = np.zeros(1, CAMERA_DTYPE)
        lens = np.zeros(1, LENS_DTYPE)
        _check(lib().pt_scene_frame(self._h, C.c_int(frame), _p(g), _p(m), _p(cam), _p(lens)))
        return g, m, cam, (float(lens["aperture"][0]), float(lens["focal_distance"][0]))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().pt_scene_free(self._h)
            self._h = C.c_void_p()

    __del__ = close


def save_image(rgb, width, height, image_name, frame=0, force_png=True):
    """runCuda's save path (src/main.cpp:118-139) + image::saveImageRGB (src/image.cpp:46-88)."""
    rgb = _arr(rgb, np.float32)
    assert rgb.size == width * height * 3
    out = C.create_string_buffer(1024)
    _check(lib().pt_save_image(_p(rgb), C.c_int(width), C.c_int(height), str(image_name).encode(), C.c_int(frame),
                               C.c_int(1 if force_png else 0), out, C.c_int(1024)))
    return out.value.decode()


def image_to_rgb8(rgb, width, height):
    rgb = _arr(rgb, np.float32)
    out = np.empty((height, width, 3), np.uint8)
    _check(lib().pt_image_to_rgb8(_p(rgb), C.c_int(width), C.c_int(height), _p(out)))
    return out


def render_frame(geoms, materials, camera, spp, max_depth, seed=0, lens=None, device=0, wavefront_paths=None):
    """Convenience: one whole render -> (mean image (H*W,3) float32, paths, segments, live, gpu_ms)."""
    with Context(geoms, materials, camera, lens, device) as ctx:
        if wavefront_paths:
            ctx.set_wavefront_paths(wavefront_paths)
        ctx.render(0, spp, max_depth, seed)
        img = ctx.download_mean(spp)
        paths, segs, live = ctx.counters()
        return img, paths, segs, live, ctx.last_render_ms()
