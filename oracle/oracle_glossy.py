"""TEST INFRASTRUCTURE ONLY: ctypes bindings for oracle/libpt_oracle_glossy.so, the C restatement (pt_oracle.c) with
subsurface scattering (pt_oracle_medium.c) extended by glossy reflection (pt_oracle_glossy.c, DESIGN.md 4).

Only tests/, __graft_entry__.build() and oracle/gen_glossy_golden.py import this.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle_medium import OracleMedium
from oracle_py import HERE, _f32, _p

GLOSSY_SO = os.path.join(HERE, "libpt_oracle_glossy.so")
_SRCS = [os.path.join(HERE, f) for f in ("pt_oracle_glossy.c", "pt_oracle_glossy.h", "pt_oracle_medium.c",
                                          "pt_oracle_medium.h", "pt_oracle.c", "pt_oracle.h")]


def build_oracle_glossy(force=False):
    """Compile pt_oracle_glossy.c (which includes pt_oracle_medium.c and pt_oracle.c) with the restatement's flags"""
    if not force and os.path.exists(GLOSSY_SO) and os.path.getmtime(GLOSSY_SO) >= max(os.path.getmtime(s) for s in _SRCS):
        return
    tmp = GLOSSY_SO + ".tmp.%d" % os.getpid()
    try:
        subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                               "-Wall", "-Wextra", "-o", tmp, _SRCS[0], "-lm"])
        os.replace(tmp, GLOSSY_SO)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


class OracleGlossy(OracleMedium):
    """Oracle with glossy reflection: make_scene(..., glossy=True) samples the Phong lobe of SPECEX > 0 reflectors
    (or_render_ext); every other function is the medium library's own (this library contains all of it)."""

    def __init__(self):
        super().__init__()
        build_oracle_glossy()
        medium = self.lib
        L = self.lib = C.CDLL(GLOSSY_SO)
        for name in ("or_hash", "or_sphereIntersectionTest", "or_boxIntersectionTest", "or_u01", "or_render_sss",
                     "or_render_ex", "or_max_threads", "or_refract", "or_log"):
            f, g = getattr(L, name), getattr(medium, name)
            f.restype = g.restype
            if g.argtypes is not None:
                f.argtypes = g.argtypes
        L.or_render_ext.restype = C.c_double
        L.or_render_ext.argtypes = [C.c_void_p, C.c_int, C.c_int] + medium.or_render_sss.argtypes[2:]

    def sample_glossy(self, normal, incident, exponent, u):
        """the glossy lobe: outward normal (n,3), incident direction (n,3), SPECEX (n,), u = (n,2) -> direction (n,3)"""
        nn, d = _f32(normal).reshape(-1, 3), _f32(incident).reshape(-1, 3)
        e, uu = _f32(exponent).ravel(), _f32(u).reshape(-1, 2)
        n = e.size
        assert nn.shape[0] == n and d.shape[0] == n and uu.shape[0] == n
        out = np.zeros((n, 3), np.float32)
        self.lib.or_sample_glossy_batch(C.c_int(n), _p(nn), _p(d), _p(e), _p(uu), _p(out))
        return out

    def make_scene(self, geoms, materials, cam, lens=(0.0, 0.0), direct_lighting=False, subsurface=False, glossy=False):
        sc = super().make_scene(geoms, materials, cam, lens, direct_lighting, subsurface)
        sc._glossy = 1 if glossy else 0
        return sc

    def render(self, scene, first_sample, n_samples, max_depth, seed, pix_begin=0, pix_end=None, threads=0,
               sum_rgb=None, path_loop="ext"):
        """OracleMedium.render through or_render_ext (path_loop="ext"), or_render_sss ("sss") or or_render_ex ("ex")"""
        if path_loop != "ext":
            return super().render(scene, first_sample, n_samples, max_depth, seed, pix_begin, pix_end, threads, sum_rgb,
                                  path_loop)
        W, H = int(scene.cam.resolution[0]), int(scene.cam.resolution[1])
        if pix_end is None:
            pix_end = W * H
        if sum_rgb is None:
            sum_rgb = np.zeros((W * H, 3), np.float32)
        live = np.zeros(64, np.uint64)
        shadow = C.c_uint64(0)
        secs = self.lib.or_render_ext(C.byref(scene), getattr(scene, "_subsurface", 0), getattr(scene, "_glossy", 0),
                                      first_sample, n_samples, max_depth, seed, pix_begin, pix_end, _p(sum_rgb), _p(live),
                                      threads, C.byref(shadow))
        self.last_shadow_rays = int(shadow.value)
        return sum_rgb, live[:max_depth].copy(), float(secs)
