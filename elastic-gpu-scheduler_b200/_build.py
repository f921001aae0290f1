"""In-tree builds: libegs.so (CUDA, sm_100a) and libegs_synth.so (plain C harness helper)."""
from __future__ import annotations

import glob
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
LIBEGS = os.path.join(LIBDIR, "libegs.so")
LIBSYNTH = os.path.join(LIBDIR, "libegs_synth.so")

NVCC_FLAGS = (["-DEGS_RESOLVE_PROF"] if os.environ.get("EGS_RESOLVE_PROF") else []) + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _stale(target: str, sources) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: libegs cannot be built")
    return p


def build_libegs(force: bool = False, verbose: bool = False) -> str:
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
                  [os.path.join(ROOT, "include", "egs.h")])
    if force or _stale(LIBEGS, srcs):
        os.makedirs(LIBDIR, exist_ok=True)
        cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + \
              ["-o", LIBEGS, os.path.join(CSRC, "egs_api.cu"), "-ldl"]
        subprocess.check_call(cmd)
    return LIBEGS


LIBPROF = os.path.join(LIBDIR, "libegs_prof.so")


def build_prof(force: bool = False) -> str:
    """PROFILING ONLY (tools/gpu_round.sh, tools/prof_sections.py with EGS_LIB=libegs_prof.so): libegs with the
    resolver's clock64 section counters compiled in (-DEGS_RESOLVE_PROF).  Not part of build_all."""
    srcs = sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")) +
                  [os.path.join(ROOT, "include", "egs.h")])
    if force or _stale(LIBPROF, srcs):
        os.makedirs(LIBDIR, exist_ok=True)
        flags = [f for f in NVCC_FLAGS if f != "-DEGS_RESOLVE_PROF"]
        subprocess.check_call([nvcc_path(), "-DEGS_RESOLVE_PROF"] + flags + ["-o", LIBPROF, os.path.join(CSRC, "egs_api.cu"), "-ldl"])
    return LIBPROF


def build_synth(force: bool = False) -> str:
    src = os.path.join(CSRC, "egs_synth.c")
    if force or _stale(LIBSYNTH, [src]):
        os.makedirs(LIBDIR, exist_ok=True)
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-o", LIBSYNTH, src])
    return LIBSYNTH


LIBHOST = os.path.join(LIBDIR, "libegs_host.so")


def build_host(force: bool = False) -> str:
    """C++ mirror of the reference's ResourceScheduler plugin interface over the C ABI."""
    hdir = os.path.join(CSRC, "host")
    srcs = sorted(glob.glob(os.path.join(hdir, "*.cc")) + glob.glob(os.path.join(hdir, "*.h")) +
                  [os.path.join(ROOT, "include", "egs.h")])
    build_libegs(force)
    if force or _stale(LIBHOST, srcs + [LIBEGS]):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", LIBHOST] +
                              sorted(glob.glob(os.path.join(hdir, "*.cc"))) +
                              ["-L" + LIBDIR, "-legs", "-Wl,-rpath,$ORIGIN"])
    return LIBHOST


LIBDEVHOST = os.path.join(LIBDIR, "libegs_devhost.so")


def build_devhost(force: bool = False) -> str:
    """The kernels' integer arithmetic (csrc/egs_device.cuh) compiled for the host: CPU-side tests only."""
    src = os.path.join(CSRC, "host_test", "device_on_host.cu")
    deps = [src, os.path.join(CSRC, "egs_device.cuh"), os.path.join(ROOT, "include", "egs.h")]
    if force or _stale(LIBDEVHOST, deps):
        os.makedirs(LIBDIR, exist_ok=True)
        subprocess.check_call([nvcc_path()] + NVCC_FLAGS + ["-o", LIBDEVHOST, src])
    return LIBDEVHOST


SHIM_DOUBLE = os.path.join(ROOT, "integration", "_build", "shim_double")


def build_shim_double(force: bool = False) -> str:
    """C test double of the Go shim (integration/shim_double.c): same libegs calls, same order."""
    src = os.path.join(ROOT, "integration", "shim_double.c")
    build_libegs(force)
    if force or _stale(SHIM_DOUBLE, [src, LIBEGS, os.path.join(ROOT, "include", "egs.h")]):
        os.makedirs(os.path.dirname(SHIM_DOUBLE), exist_ok=True)
        # rpath relative to the binary, so a built tree still runs after it is copied or moved
        rpath = os.path.join("$ORIGIN", os.path.relpath(LIBDIR, os.path.dirname(SHIM_DOUBLE)))
        subprocess.check_call(["gcc", "-O2", "-o", SHIM_DOUBLE, src, "-L" + LIBDIR, "-legs", "-Wl,-rpath," + rpath])
    return SHIM_DOUBLE


def build_all(force: bool = False) -> None:
    build_synth(force)
    build_libegs(force)
    build_host(force)
    build_devhost(force)
    build_shim_double(force)
