"""TEST INFRASTRUCTURE ONLY: ctypes bindings for oracle/libpt_oracle_roulette.so, the C restatement (pt_oracle.c) with
subsurface scattering (pt_oracle_medium.c) and glossy reflection (pt_oracle_glossy.c) extended by Russian roulette
(pt_oracle_roulette.c, DESIGN.md 4).

Only tests/ and __graft_entry__.build() import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_glossy import OracleGlossy
from oracle_py import HERE, _p

ROULETTE_SO = os.path.join(HERE, "libpt_oracle_roulette.so")
_SRCS = [os.path.join(HERE, f) for f in ("pt_oracle_roulette.c", "pt_oracle_roulette.h", "pt_oracle_glossy.c",
                                          "pt_oracle_glossy.h", "pt_oracle_medium.c", "pt_oracle_medium.h", "pt_oracle.c",
                                          "pt_oracle.h")]


def build_oracle_roulette(force=False):
    """Compile pt_oracle_roulette.c (which includes pt_oracle_glossy.c and with it the rest) with the restatement's flags"""
    if not force and os.path.exists(ROULETTE_SO) and os.path.getmtime(ROULETTE_SO) >= max(os.path.getmtime(s) for s in _SRCS):
        return
    tmp = ROULETTE_SO + ".tmp.%d" % os.getpid()
    try:
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                               "-Wall", "-Wextra", "-o", tmp, _SRCS[0], "-lm"])
        os.replace(tmp, ROULETTE_SO)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


class OracleRoulette(OracleGlossy):
    """Oracle with Russian roulette: make_scene(..., roulette=k) ends paths at random from depth k (or_render_rr); every
    other function is the glossy library's own (this library contains all of it)."""

    def __init__(self):
        super().__init__()
        build_oracle_roulette()
        glossy = self.lib
        L = self.lib = C.CDLL(ROULETTE_SO)
        for name in ("or_hash", "or_sphereIntersectionTest", "or_boxIntersectionTest", "or_u01", "or_render_sss",
                     "or_render_ex", "or_render_ext", "or_max_threads", "or_refract", "or_log", "or_sample_glossy_batch"):
            f, g = getattr(L, name), getattr(glossy, name)
            f.restype = g.restype
            if g.argtypes is not None:
                f.argtypes = g.argtypes
        L.or_render_rr.restype = C.c_double
        L.or_render_rr.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + glossy.or_render_ext.argtypes[3:]
        L.or_roulette.restype = C.c_int
        L.or_roulette.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]

    def roulette(self, seed, pixel, sample, depth, thr):
        """one roulette step on throughput thr (3,) -> (survives, the throughput it goes on with)"""
        t = np.array(thr, np.float32).reshape(3).copy()
        ok = self.lib.or_roulette(seed, pixel, sample, depth, _p(t))
        return bool(ok), t

    def make_scene(self, geoms, materials, cam, lens=(0.0, 0.0), direct_lighting=False, subsurface=False, glossy=False,
                   roulette=0):
        sc = super().make_scene(geoms, materials, cam, lens, direct_lighting, subsurface, glossy)
        sc._roulette = int(roulette)
        return sc

    def render(self, scene, first_sample, n_samples, max_depth, seed, pix_begin=0, pix_end=None, threads=0,
               sum_rgb=None, path_loop="rr"):
        """OracleGlossy.render through or_render_rr (path_loop="rr"), or_render_ext ("ext"), or_render_sss ("sss") or
        or_render_ex ("ex")"""
        if path_loop != "rr":
            return super().render(scene, first_sample, n_samples, max_depth, seed, pix_begin, pix_end, threads, sum_rgb,
                                  path_loop)
        W, H = int(scene.cam.resolution[0]), int(scene.cam.resolution[1])
        if pix_end is None:
            pix_end = W * H
        if sum_rgb is None:
            sum_rgb = np.zeros((W * H, 3), np.float32)
        live = np.zeros(64, np.uint64)
        shadow = C.c_uint64(0)
        secs = self.lib.or_render_rr(C.byref(scene), getattr(scene, "_subsurface", 0), getattr(scene, "_glossy", 0),
                                     getattr(scene, "_roulette", 0), first_sample, n_samples, max_depth, seed, pix_begin,
                                     pix_end, _p(sum_rgb), _p(live), threads, C.byref(shadow))
        self.last_shadow_rays = int(shadow.value)
        return sum_rgb, live[:max_depth].copy(), float(secs)
