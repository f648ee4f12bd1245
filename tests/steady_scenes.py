"""Scenes and frame sizes for the steady-state parity tests (tests/test_oracle_steady_scenes.py on the CPU,
tests/test_gpu_steady_state.py).

The bounce kernels are persistent: warps take tickets of 4 units of 32 paths from a counter, and the hierarchy kernel
takes pools of up to 1 024 paths.  A frame only exercises the state they run in for real (queues that cycle many times,
staging across tickets, full pools, deferred lists carried from pool to pool) when it gives every warp many tickets, so
the frames here are sized from the device's SM count.  Exact-scan fallbacks and deferred exact traversals are forced by
geometry: a geom and its exact copy (same transform bits) tie on every bound, so the filter cannot decide between them
and the lower geom index must win; the copies carry different materials, so a wrong tie-break shows in the pixels."""
import math

import numpy as np

from medium_scenes import material
from roulette_scenes import closed_room
from scenes_for_tests import build_geom, random_scene

# Upper bound on the resident warps of every bounce kernel: 4 CTAs x 8 warps per SM (k_bounce; k_bounce_q runs 3 x 8).
WARPS_PER_SM = 4 * 8
TICKET_PATHS = 4 * 32  # one ticket: 4 units of 32 paths
POOL_PATHS = 1024      # k_bounce_bvh's largest pool

# Shares of a wavefront still alive that the frame sizes below are computed for (measured with the oracle at small size,
# tests/test_oracle_steady_scenes.py): at depth 4 in steady_room with every switch on and roulette from depth 1, and at
# depth 1 in steady_hierarchy (where only paths that end on the light are gone).
ROOM_KEEP_DEPTH4 = 0.85
HIERARCHY_KEEP_DEPTH1 = 0.98


def bounce_warps(sms):
    return WARPS_PER_SM * sms


def tickets_per_warp(live, sms, wavefronts=1):
    """tickets per warp that each depth's live count gives, per wavefront"""
    return np.asarray(live, np.float64) / wavefronts / (TICKET_PATHS * bounce_warps(sms))


def room_side(sms, tickets=6, keep=ROOM_KEEP_DEPTH4):
    """side of a square frame whose W*H-path wavefront still holds `tickets` tickets per warp at depth 4"""
    need = tickets * TICKET_PATHS * bounce_warps(sms) / keep
    return 32 * math.ceil(math.sqrt(need) / 32)


def hierarchy_side(sms, spp=2, keep=HIERARCHY_KEEP_DEPTH1):
    """side of a square frame whose spp-sample wavefront keeps k_bounce_bvh's pools full size (bvh_take_pool: at least
    2 * warps * 1024 paths left) at depths 0 and 1"""
    need = 2 * bounce_warps(sms) * POOL_PATHS / spp / keep
    return 32 * math.ceil(math.sqrt(need) / 32)


def _room_materials(pt, walls):
    """closed_room's materials (walls, light, diffuse sphere) and the ones added here: twin sphere, interior cube, twin
    cube, medium, glossy"""
    m = np.zeros(8, pt.MATERIAL_DTYPE)
    m[:3] = walls
    m[1]["emittance"] = 6.0
    m[2]["color"] = (0.5, 0.99, 0.6)
    m[3] = material(pt, color=(0.99, 0.3, 0.2))                          # twin of the sphere: red instead of green
    m[4] = material(pt, color=(0.3, 0.4, 0.99))                          # interior cube: blue
    m[5] = material(pt, color=(0.99, 0.9, 0.3))                          # its twin: yellow
    m[6] = material(pt, color=(0.99, 0.99, 0.99), refr=1.0, ior=1.3, scatter=1.0, rsct=2.0,
                    absorption=(0.01, 0.03, 0.06))                        # medium
    m[7] = material(pt, color=(0.9, 0.9, 0.9), spec=(0.99, 0.9, 0.85))   # glossy
    m[7]["hasReflective"], m[7]["specularExponent"] = 1.0, 40.0
    return m


def steady_room(pt, camera, w, h):
    """closed_room (albedo below 1 so the roulette draws, a small light under the ceiling) with a medium sphere, a glossy
    sphere, an interior cube, and an exact copy of the diffuse sphere and of the cube, each with its own material.
    13 geoms: the few-geom kernels (pair scan).  Twin pairs: (7, 8) and (9, 10)."""
    g0, m0, cam = closed_room(pt, camera, w, h, albedo=0.99)
    g0[6] = build_geom(pt, 1, 1, (0, 2.8, 0), (0, 0, 0), (1.2, .1, 1.2))  # a smaller light: fewer paths end on it
    g = np.zeros(13, pt.GEOM_DTYPE)
    g[:8] = g0
    g[7] = build_geom(pt, 0, 2, (-0.9, -1.2, -1.0), (0, 0, 0), (1.6, 1.6, 1.6))
    g[8] = g[7]
    g[8]["materialid"] = 3
    g[9] = build_geom(pt, 1, 4, (0.9, -1.4, -0.6), (10, 35, 5), (1.2, 1.2, 1.2))
    g[10] = g[9]
    g[10]["materialid"] = 5
    g[11] = build_geom(pt, 0, 6, (0.8, 0.6, -1.4), (0, 0, 0), (1.4, 1.4, 1.4))
    g[12] = build_geom(pt, 0, 7, (-1.0, 0.7, -1.6), (0, 0, 0), (1.3, 1.3, 1.3))
    return g, _room_materials(pt, m0), cam


def steady_hierarchy(pt, camera, w, h):
    """a closed room with 40 geoms (the hierarchy kernels): 21 small random interior geoms, a medium and a glossy
    sphere, two twin pairs (the second candidate settles their hits) and two triplets (three candidates tie: the exact
    traversal settles them), every copy with its own material.  Returns (geoms, materials, camera, twins, triplets)
    with the index groups of the copies."""
    g0, m0, cam = closed_room(pt, camera, w, h, albedo=0.99)
    g0[6] = build_geom(pt, 1, 1, (0, 2.8, 0), (0, 0, 0), (1.2, .1, 1.2))
    m = np.concatenate([_room_materials(pt, m0), np.zeros(4, pt.MATERIAL_DTYPE)])
    m[8] = material(pt, color=(0.2, 0.99, 0.9))
    m[9] = material(pt, color=(0.99, 0.2, 0.9))
    m[10] = material(pt, color=(0.6, 0.6, 0.99))
    m[11] = material(pt, color=(0.99, 0.6, 0.1))
    rnd = random_scene(pt, 21, 5, extent=1.8, smin=0.15, smax=0.45, offset=(0, 0, -0.8))
    rnd["materialid"] = np.array([0, 2, 4, 10])[np.arange(21) % 4]
    parts = [g0[:7], rnd]
    groups = []

    def copies(base, mats):
        first = sum(len(p) for p in parts)
        c = np.zeros(len(mats), pt.GEOM_DTYPE)
        for i, mi in enumerate(mats):
            c[i] = base
            c[i]["materialid"] = mi
        parts.append(c)
        groups.append(list(range(first, first + len(mats))))

    copies(build_geom(pt, 0, 2, (-1.1, -1.3, -1.2), (0, 0, 0), (1.3, 1.3, 1.3)), [2, 3])
    copies(build_geom(pt, 1, 4, (1.1, -1.5, -0.9), (15, 30, 0), (1.0, 1.0, 1.0)), [4, 5])
    copies(build_geom(pt, 0, 8, (1.2, 0.9, -1.7), (0, 0, 0), (1.1, 1.1, 1.1)), [8, 9, 11])
    copies(build_geom(pt, 1, 10, (-1.3, 1.0, -1.9), (20, 10, 40), (0.9, 0.9, 0.9)), [10, 3, 5])
    parts.append(np.array([build_geom(pt, 0, 6, (0.0, -0.2, -2.0), (0, 0, 0), (1.2, 1.2, 1.2)),
                           build_geom(pt, 0, 7, (0.0, 1.6, -1.2), (0, 0, 0), (0.9, 0.9, 0.9))], pt.GEOM_DTYPE))
    g = np.concatenate(parts)
    twins = [grp for grp in groups if len(grp) == 2]
    triplets = [grp for grp in groups if len(grp) == 3]
    return g, m, cam, twins, triplets
