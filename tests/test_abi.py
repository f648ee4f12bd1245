"""The C-ABI shared library: builds without a GPU, loads, exports every symbol the headers declare, and fails
loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    syms = set()
    for hdr in ("pt_b200.h", "pt_compat.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        text = re.sub(r"//[^\n]*", "", text)
        syms |= set(re.findall(r"\b(pt_[a-z0-9_]+)\s*\(", text))
    return syms


def test_library_exports_every_declared_symbol(pt):
    lib = pt.lib()
    syms = declared_symbols()
    assert len(syms) >= 35
    missing = [s for s in sorted(syms) if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.pt_abi_version() == 1


def test_up_to_date_build_writes_nothing(pt, monkeypatch):
    """a built tree may be read-only: loading it must not take the build lock (which creates a file in the package)"""
    pt.lib()

    def no_lock():
        raise AssertionError("build() took the lock although nothing was stale")
    monkeypatch.setattr(pt.build, "_locked", no_lock)
    assert pt.build.build() == pt.LIB_PATH


def test_cudaRaytraceCore_symbol_has_the_reference_mangling(pt):
    """same C++ symbol as the reference's src/raytraceKernel.h:17 declaration produces"""
    out = subprocess.check_output(["nm", "-D", "--defined-only", pt.LIB_PATH], text=True)
    assert "_Z16cudaRaytraceCoreP6uchar4P6cameraiiP8materialiP4geomi" in out


def test_no_oracle_in_the_product():
    """the product never routes through the oracle or any CPU fallback"""
    pkg = os.path.join(ROOT, "project3-pathtracer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle_py" not in text and "pt_oracle" not in text and "libpt_oracle" not in text, f
    out = subprocess.check_output(["ldd", os.path.join(pkg, "libpt_b200.so")], text=True)
    assert "oracle" not in out


def test_compute_entry_points_fail_loudly_without_a_gpu(pt, sample_scene):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        pytest.skip("a GPU is present")
    with pytest.raises(pt.PtError) as e:
        pt.Context(sample_scene["geoms"], sample_scene["materials"], sample_scene["camera"])
    assert "cuda" in str(e.value).lower()
    with pytest.raises(pt.PtError):
        pt.compact_u32(np.arange(4, dtype=np.uint32), np.ones(4, np.uint8))
    with pytest.raises(pt.PtError):
        pt.random_points_on_geom(sample_scene["geoms"][0:1], [1.0])
    with pytest.raises(pt.PtError):
        pt.random_directions_in_sphere([0.5], [0.5])
    with pytest.raises(pt.PtError):
        pt.calculate_transmission([[1, 1, 1]], [1.0])
    with pytest.raises(pt.PtError):
        pt.reference_stub_image(8, 8, 1)


def test_argument_validation(pt):
    lib = pt.lib()
    n = C.c_int()
    assert lib.pt_device_count(None) == -1  # PT_ERR_INVALID
    assert b"NULL" in lib.pt_last_error()
    assert lib.pt_scene_load(None, 0, None) == -1
    assert lib.pt_context_destroy(None) == 0
    assert lib.pt_compat_set_trace_depth(0) == -1 and lib.pt_compat_set_trace_depth(8) == 0
