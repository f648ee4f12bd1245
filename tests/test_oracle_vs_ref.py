"""Pins the C restatement against the reference's own functions (oracle/_ref/libptref.so) on large seeded ray sets.
Runs wherever oracle/_ref has been built (the build container; the prebuilt .so also travels to the GPU box)."""
import numpy as np
import pytest

from conftest import same_bits
from oracle_py import Ref

pytestmark = pytest.mark.skipif(not Ref.available(), reason="oracle/_ref not built (needs the reference checkout at build time: PT_REFERENCE_DIR, default /root/reference)")


@pytest.fixture(scope="module")
def ref():
    return Ref()


def test_sphere_test_bit_exact_on_random_rays(oracle, ref, sample_scene):
    rng = np.random.default_rng(17)
    g = sample_scene["geoms"]
    hits = 0
    for gi in range(len(g)):
        n = 4000
        o = rng.uniform(-8, 14, (n, 3)).astype(np.float32)
        tgt = g[gi]["translation"] + rng.normal(0, 0.6, (n, 3)).astype(np.float32) * g[gi]["scale"]
        d = (tgt - o).astype(np.float32)
        d[: n // 2] /= np.linalg.norm(d[: n // 2], axis=1, keepdims=True)  # half normalised, half not
        o[-500:] = (g[gi]["translation"] + rng.uniform(-0.4, 0.4, (500, 3)) * g[gi]["scale"]).astype(np.float32)
        t1, p1, n1 = oracle.intersect_one(g[gi], 0, o, d)
        t2, p2, n2 = ref.intersect_one(g[gi], 0, o, d)
        assert same_bits(t1, t2)
        h = t2 > 0
        hits += int(h.sum())
        assert same_bits(p1[h], p2[h]) and same_bits(n1[h], n2[h])
    assert hits > 5000


def test_hemisphere_hash_radiuses(oracle, ref, sample_scene):
    rng = np.random.default_rng(23)
    nn = rng.normal(size=(5000, 3)).astype(np.float32)
    nn /= np.linalg.norm(nn, axis=1, keepdims=True)
    x1, x2 = rng.random(5000, dtype=np.float32), rng.random(5000, dtype=np.float32)
    assert same_bits(oracle.hemisphere(nn, x1, x2, ref=True), ref.hemisphere(nn, x1, x2))
    for a in rng.integers(0, 2**32, 200):
        assert oracle.hash(int(a)) == ref.hash(int(a))
    for g in sample_scene["geoms"]:
        assert same_bits(oracle.getRadiuses(g), ref.getRadiuses(g))
