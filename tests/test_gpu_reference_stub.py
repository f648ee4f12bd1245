"""GPU parity against the reference ITSELF: oracle/_ref/libptref_gpu.so is the reference's own src/raytraceKernel.cu
compiled for sm_100a (oracle/ref_kernel_shim.cu includes it from where it lies).  Its renderer is the stub the
reference ships, so what can be compared is what it does implement: the per-pixel noise of raytraceRay /
generateRandomNumberFromThread (:29-36, 93-104) and the 8-bit conversion of sendImageToPBO (:58-89).  Bit-exact."""
import json
import os

import numpy as np
import pytest

from conftest import GOLD, f32, same_bits, with_resolution

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def refgpu():
    from oracle_py import RefGpu
    if not RefGpu.available():
        pytest.skip("oracle/_ref/libptref_gpu.so not built (needs the reference checkout at build time: PT_REFERENCE_DIR, default /root/reference)")
    return RefGpu()


@pytest.mark.parametrize("W,H,k", [(96, 96, 1), (160, 64, 7), (800, 800, 5000)])
def test_stub_image_equals_the_reference_kernel(pt, oracle, refgpu, W, H, k):
    img_ref, _ = refgpu.cudaRaytraceCore(W, H, k)
    ours = pt.reference_stub_image(W, H, k, pt.STUB_ORDER_DEVICE)
    assert same_bits(ours, img_ref)
    # the reference overwrites whatever renderCam->image held (no accumulation in the stub)
    junk = np.random.default_rng(0).random((W * H, 3)).astype(np.float32)
    again, _ = refgpu.cudaRaytraceCore(W, H, k, image=junk)
    assert same_bits(again, img_ref)
    # the host build of the same function draws in the opposite order; oracle and CUDA agree on both
    assert same_bits(pt.reference_stub_image(W, H, k, pt.STUB_ORDER_HOST), oracle.noise_image(W, H, float(k), True))
    assert same_bits(ours, oracle.noise_image(W, H, float(k), False))


def test_stub_image_equals_the_stored_reference_output(pt):
    """the same comparison against the reference's own output stored in tests/golden/sampling_vectors.json (its host
    build of generateRandomNumberFromThread), so it runs without a build of the reference"""
    with open(os.path.join(GOLD, "sampling_vectors.json")) as f:
        cases = json.load(f)["ref_noise_host"]
    for k in cases:
        want = f32(k["rgb"]).reshape(-1, 3)
        assert same_bits(pt.reference_stub_image(k["W"], k["H"], int(k["time"]), pt.STUB_ORDER_HOST), want)
        # the device build draws the same three numbers in the opposite order (stored host output only; the device
        # order itself is compared with the reference's kernel by test_stub_image_equals_the_reference_kernel)
        assert same_bits(pt.reference_stub_image(k["W"], k["H"], int(k["time"]), pt.STUB_ORDER_DEVICE), want[:, ::-1])


def test_resolve_rgba8_equals_sendImageToPBO(pt, refgpu, sample_scene):
    """our 8-bit resolve of the reference's image == the PBO the reference's own kernel wrote from it"""
    W, H = 128, 64
    img_ref, pbo_ref = refgpu.cudaRaytraceCore(W, H, 3)
    cam = with_resolution(sample_scene["camera"], W, H)
    with pt.Context(sample_scene["geoms"], sample_scene["materials"], cam) as c:
        for scale in (1.0, 1.7, 0.25):  # values above 1 exercise the clamp at 255
            c.upload_sum(img_ref * np.float32(scale))
            got = c.resolve_rgba8(1)
            want = np.minimum(img_ref * np.float32(scale) * np.float32(255.0), np.float32(255.0)).astype(np.uint8)
            assert (got[:, :3] == want).all() and (got[:, 3] == 0).all()
            if scale == 1.0:
                assert (got == pbo_ref).all()


def test_cudaRaytraceCore_drop_in_equals_the_reference_entry_point(pt, refgpu, sample_scene):
    """the same call -- cudaRaytraceCore(pbo, camera, frame, iterations, ...) -- into the reference's own library and into
    ours (stub mode): renderCam->image and the device PBO come back identical, byte for byte"""
    import importlib
    import torch
    compat = importlib.import_module("project3-pathtracer_b200.compat")
    W, H = 96, 64
    cam = with_resolution(sample_scene["camera"], W, H)
    rs = compat.RefScene([(sample_scene["geoms"], cam)], sample_scene["materials"], iterations=3)
    compat.reset(); compat.set_exit_on_error(False); compat.set_reference_stub(True)
    try:
        for k in (1, 2, 9):
            pbo = torch.full((W * H * 4,), 0xAB, dtype=torch.uint8, device="cuda")
            compat.cudaRaytraceCore(pbo.data_ptr(), rs.camera, 0, k, rs.materials, len(rs.materials), rs.geoms, len(rs.geoms))
            assert compat.last_status() == 0
            img_ref, pbo_ref = refgpu.cudaRaytraceCore(W, H, k)
            assert same_bits(rs.image, img_ref)
            assert (pbo.cpu().numpy().reshape(-1, 4) == pbo_ref).all()
    finally:
        compat.set_reference_stub(False)
        compat.reset()
