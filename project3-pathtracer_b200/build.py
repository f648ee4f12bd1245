"""Build libpt_b200.so (CUDA kernels + C ABI + host loader / image writer / compat shim) and the headless
driver `pt_render`, in-tree, for sm_100a.  No GPU is needed to build (nvcc cross-compiles)."""
import contextlib
import fcntl
import glob
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
ROOT = os.path.dirname(PKG)
LIB = os.path.join(PKG, "libpt_b200.so")
DRIVER = os.path.join(PKG, "pt_render")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
# -fmad=false + IEEE sqrt/div (nvcc defaults): the arithmetic contract of csrc/pt_device.cuh
NVCC_FLAGS = ARCH + ["-lineinfo", "-O3", "-std=c++17", "-fmad=false", "-Xcompiler", "-fPIC,-ffp-contract=off,-O2"]


def nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: the B200 path tracer cannot be built (there is no CPU fallback)")
    return exe


def _sources():
    cu = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    cpp = sorted(p for p in glob.glob(os.path.join(CSRC, "*.cpp")) if os.path.basename(p) != "pt_main.cpp")
    return cu, cpp


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


@contextlib.contextmanager
def _locked():
    """One builder at a time: under torchrun every rank imports the package (and may find it stale) at once."""
    fd = os.open(os.path.join(PKG, ".build.lock"), os.O_CREAT | os.O_RDWR, 0o644)
    try:
        fcntl.flock(fd, fcntl.LOCK_EX)
        yield
    finally:
        fcntl.flock(fd, fcntl.LOCK_UN)
        os.close(fd)


def _stale_outputs(force=False):
    """(cu sources, cpp sources, library stale, driver stale): the one rule for what a build has to redo"""
    cu, cpp = _sources()
    hdr = glob.glob(os.path.join(CSRC, "*.h")) + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(
        os.path.join(ROOT, "include", "*.h"))
    lib = force or _stale(LIB, cu + cpp + hdr + [os.path.abspath(__file__)])
    main = os.path.join(CSRC, "pt_main.cpp")
    driver = os.path.exists(main) and (lib or _stale(DRIVER, [main, LIB]))
    return cu, cpp, lib, driver


def build(force=False, verbose=False):
    """Build what is stale.  Serialised by a file lock; outputs are written to a temporary name and renamed, so a
    concurrent dlopen never sees a half-written file.  An up-to-date build takes no lock and writes nothing, so a
    built tree can be used read-only."""
    if not any(_stale_outputs(force)[2:]):
        return LIB
    with _locked():
        return _build(force, verbose)


def _build(force, verbose):
    cu, cpp, lib, driver = _stale_outputs(force)  # again under the lock: another process may have built meanwhile
    if lib:
        tmp = LIB + ".tmp.%d" % os.getpid()
        cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + [
            "-I", os.path.join(ROOT, "include"), "-shared", "-o", tmp] + cu + cpp + ["-lz"]
        try:
            subprocess.check_call(cmd)
            os.replace(tmp, LIB)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    if driver:
        main = os.path.join(CSRC, "pt_main.cpp")
        tmp = DRIVER + ".tmp.%d" % os.getpid()
        try:
            subprocess.check_call(["g++", "-std=c++17", "-O2", "-pthread", "-I", os.path.join(ROOT, "include"), main, "-o", tmp,
                                   "-L", PKG, "-lpt_b200", "-Wl,-rpath,$ORIGIN"])
            os.replace(tmp, DRIVER)
        finally:
            if os.path.exists(tmp):
                os.remove(tmp)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
