"""TEST INFRASTRUCTURE ONLY: ctypes bindings for oracle/libpt_oracle_medium.so, the C restatement (pt_oracle.c) extended
by subsurface scattering (pt_oracle_medium.c, DESIGN.md 4).

Only tests/, __graft_entry__.build() and oracle/gen_medium_golden.py import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_py import HERE, Oracle, _f32, _p

MEDIUM_SO = os.path.join(HERE, "libpt_oracle_medium.so")
_SRCS = [os.path.join(HERE, f) for f in ("pt_oracle_medium.c", "pt_oracle_medium.h", "pt_oracle.c", "pt_oracle.h")]


def build_oracle_medium(force=False):
    """Compile pt_oracle_medium.c (which includes pt_oracle.c) with the restatement's flags (oracle/Makefile)."""
    if not force and os.path.exists(MEDIUM_SO) and os.path.getmtime(MEDIUM_SO) >= max(os.path.getmtime(s) for s in _SRCS):
        return
    tmp = MEDIUM_SO + ".tmp.%d" % os.getpid()
    try:
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                               "-Wall", "-Wextra", "-o", tmp, _SRCS[0], "-lm"])
        os.replace(tmp, MEDIUM_SO)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


class OracleMedium(Oracle):
    """Oracle with subsurface scattering: make_scene(..., subsurface=True) renders media (or_render_sss); every other
    function is the C restatement's own (the library contains all of pt_oracle.c)."""

    def __init__(self):
        super().__init__()
        build_oracle_medium()
        L = self.lib = C.CDLL(MEDIUM_SO)
        L.or_hash.restype = C.c_uint
        L.or_hash.argtypes = [C.c_uint]
        L.or_sphereIntersectionTest.restype = C.c_float
        L.or_boxIntersectionTest.restype = C.c_float
        L.or_u01.restype = C.c_float
        L.or_u01.argtypes = [C.c_uint32]
        L.or_render_sss.restype = C.c_double
        L.or_render_sss.argtypes = [
            C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32,
            C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
        ]
        L.or_render_ex.restype = C.c_double
        L.or_render_ex.argtypes = L.or_render_sss.argtypes[:1] + L.or_render_sss.argtypes[2:]
        L.or_max_threads.restype = C.c_int
        L.or_refract.restype = C.c_int
        L.or_log.restype = C.c_float
        L.or_log.argtypes = [C.c_float]

    def log(self, x):
        return float(self.lib.or_log(C.c_float(x)))

    def sample_medium(self, absorption, scatter, distance, u):
        """calculateScatterAndAbsorption's free flight: u = (n, 3) -> (scattered bool, s, direction (n,3), weight (n,3))"""
        a, sc = _f32(absorption).reshape(-1, 3), _f32(scatter).ravel()
        d, uu = _f32(distance).ravel(), _f32(u).reshape(-1, 3)
        n = d.size
        assert a.shape[0] == n and sc.size == n and uu.shape[0] == n
        flag, s = np.zeros(n, np.int32), np.zeros(n, np.float32)
        dirs, w = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        self.lib.or_sample_medium_batch(C.c_int(n), _p(a), _p(sc), _p(d), _p(uu), _p(flag), _p(s), _p(dirs), _p(w))
        return flag.astype(bool), s, dirs, w

    def make_scene(self, geoms, materials, cam, lens=(0.0, 0.0), direct_lighting=False, subsurface=False):
        sc = super().make_scene(geoms, materials, cam, lens, direct_lighting)
        sc._subsurface = 1 if subsurface else 0
        return sc

    def render(self, scene, first_sample, n_samples, max_depth, seed, pix_begin=0, pix_end=None, threads=0,
               sum_rgb=None, path_loop="sss"):
        """Oracle.render through or_render_sss (path_loop="sss") or the restatement's own or_render_ex ("ex")"""
        W, H = int(scene.cam.resolution[0]), int(scene.cam.resolution[1])
        if pix_end is None:
            pix_end = W * H
        if sum_rgb is None:
            sum_rgb = np.zeros((W * H, 3), np.float32)
        live = np.zeros(64, np.uint64)
        shadow = C.c_uint64(0)
        args = (first_sample, n_samples, max_depth, seed, pix_begin, pix_end, _p(sum_rgb), _p(live), threads, C.byref(shadow))
        if path_loop == "sss":
            secs = self.lib.or_render_sss(C.byref(scene), getattr(scene, "_subsurface", 0), *args)
        else:
            secs = self.lib.or_render_ex(C.byref(scene), *args)
        self.last_shadow_rays = int(shadow.value)
        return sum_rgb, live[:max_depth].copy(), float(secs)
