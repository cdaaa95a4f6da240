"""Compiles libclc_b200.so (sm_100a only) in-tree with nvcc.  No GPU is needed to build."""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libclc_b200.so")
SOURCES = ["clc_api.cu", "clc_pack.cpp"]
HEADERS = ["clc_kernels.cuh", "clc_math.cuh", "clc_lm.cuh", "clc_expand.cuh", "clc_linefit.cuh", "clc_scans.cuh", "clc_camera.cuh", "clc_upload.inl"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
    "-diag-suppress", "177",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libclc_b200.so cannot be built")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS]
    deps.append(os.path.join(PKG_DIR, "..", "include", "clc_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    extra = os.environ.get("CLC_NVCC_EXTRA", "").split()  # experiment knobs, e.g. -DCLC_THREADS=512 -DCLC_BLOCKS_PER_SM=1
    out = os.environ.get("CLC_LIB_OUT", LIB_PATH)
    cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-o", out, *[os.path.join(CSRC, s) for s in SOURCES], "-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stderr)
    return out


# ---- the C++ side: the drop-in translation unit + the end-to-end bench driver (g++, no CUDA headers needed) -----------
REPO = os.path.dirname(PKG_DIR)
DROPIN_SRC = os.path.join(PKG_DIR, "host", "LaseCamCalB200.cpp")
BENCH_SRC = os.path.join(PKG_DIR, "host", "dropin_bench.cpp")
BENCH_EXE = os.path.join(PKG_DIR, "host", "clc_dropin_bench")


def interface_include_dirs():
    """Include path of the reference interface: the reference's own include/LaseCamCalCeres.h when the environment variable
    CLC_REFERENCE_INCLUDE names a directory that holds it (a checkout of the reference's include/), else the test stand-in;
    Eigen itself is not required, its few types come from tests/stubs."""
    dirs = []
    ref = os.environ.get("CLC_REFERENCE_INCLUDE")
    if ref and os.path.exists(os.path.join(ref, "LaseCamCalCeres.h")):
        dirs.append(ref)
    dirs.append(os.path.join(REPO, "tests", "stubs"))
    dirs.append(os.path.join(REPO, "include"))
    return dirs


def cxx_command(sources, out, extra=()):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-O2", "-std=c++11", "-Wall"]
    for d in interface_include_dirs():
        cmd += ["-I", d]
    cmd += list(sources) + ["-L", PKG_DIR, "-lclc_b200", "-Wl,-rpath," + PKG_DIR, "-Wl,-rpath,$ORIGIN/..", "-pthread", *extra, "-o", out]
    return cmd


def build_dropin_bench(force: bool = False) -> str:
    deps = [DROPIN_SRC, BENCH_SRC, os.path.join(REPO, "include", "clc_b200.h"), LIB_PATH]
    if not force and os.path.exists(BENCH_EXE) and all(os.path.getmtime(d) <= os.path.getmtime(BENCH_EXE) for d in deps if os.path.exists(d)):
        return BENCH_EXE
    res = subprocess.run(cxx_command([BENCH_SRC, DROPIN_SRC], BENCH_EXE), capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("g++ failed:\n" + res.stdout + res.stderr)
    return BENCH_EXE


if __name__ == "__main__":
    print(build(force=True, verbose=True))
    print(build_dropin_bench(force=True))
