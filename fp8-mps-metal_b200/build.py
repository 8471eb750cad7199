#!/usr/bin/env python3
"""
In-tree build of the native code (no JIT cache, so the artefacts travel with the tree):

  libfp8_b200.so                      CUDA kernels + C ABI (include/fp8_b200.h), nvcc, sm_100a only
  fp8_metal.cpython-*.so              torch extension binding torch tensors to that C ABI

Usage:  python fp8-mps-metal_b200/build.py [--force] [--no-ext]

nvcc cross-compiles for sm_100a without a GPU.  Flags: -gencode arch=compute_100a,code=sm_100a
-lineinfo (so ncu's source page maps to these files) -O3.
"""

from __future__ import annotations

import argparse
import hashlib
import concurrent.futures as cf
import os
import shutil
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
# FP8B_BUILD_PROFILE=1: a second, PROFILING-ONLY library (extra kernel knobs compiled in) under profiles/tools/bin/;
# the shipped libfp8_b200.so is never built with it.  Load it with FP8B_LIB=... in the profiling scripts.
PROFILE = os.environ.get("FP8B_BUILD_PROFILE") == "1"
OBJ = os.path.join(ROOT, "profiles", "tools", "bin", "obj") if PROFILE else os.path.join(HERE, "build")
LIB = os.path.join(ROOT, "profiles", "tools", "bin", "libfp8_b200_profile.so") if PROFILE else os.path.join(HERE, "libfp8_b200.so")

CU_SOURCES = ["fp8_cast.cu", "fp8_gemv.cu", "fp8_gemv_mma.cu", "fp8_gemv_batch.cu", "fp8_gemm_simt.cu", "fp8_gemm_tcgen05.cu", "fp8_capi.cu"]
HEADERS = ["fp8_codec.cuh", "fp8_common.cuh", "fp8_mm.cuh", "fp8_async.cuh"]
# -DFP8B_PROFILE adds the GEMM's profiling knobs (per-tile clock stamps, store/TMA suppression); never in a shipped build
EXTRA_NVCC_FLAGS = (["-DFP8B_PROFILE"] + os.environ.get("FP8B_PROFILE_DEFINES", "").split()) if os.environ.get("FP8B_BUILD_PROFILE") == "1" else []
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def ext_path() -> str:
    return os.path.join(HERE, "fp8_metal" + sysconfig.get_config_var("EXT_SUFFIX"))


def _digest(paths, extra=()) -> str:
    """Content hash of source files + the command-line flags that shape the output.  Staleness is decided by
    CONTENT, not mtimes: a `git checkout` gives arbitrary mtimes, and a prebuilt .so that travelled to another box
    must be rebuilt exactly when the sources next to it differ from the ones it was built from."""
    h = hashlib.sha256()
    for x in extra:
        h.update(str(x).encode())
        h.update(b"\0")
    for p in paths:
        h.update(os.path.basename(p).encode())
        h.update(b"\0")
        with open(p, "rb") as f:
            h.update(f.read())
        h.update(b"\0")
    return h.hexdigest()


def _fresh(target: str, digest: str) -> bool:
    """`target` exists and the stamp next to it (<target>.stamp) records this digest."""
    try:
        with open(target + ".stamp") as f:
            return os.path.exists(target) and f.read().strip() == digest
    except OSError:
        return False


def _stamp(target: str, digest: str) -> None:
    with open(target + ".stamp", "w") as f:
        f.write(digest + "\n")


def _run(cmd):
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("build command failed:\n  " + " ".join(cmd) + "\n" + r.stdout)
    return r.stdout


def build_lib(force: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    sources = CU_SOURCES + (["fp8_prof.cu"] if PROFILE else [])
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(ROOT, "include", "fp8_b200.h")]
    nvcc = _nvcc()
    jobs = []
    objs = []
    stamps = []
    flags = NVCC_FLAGS + EXTRA_NVCC_FLAGS
    for src in sources:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(o)
        d = _digest([s] + hdrs, flags)
        stamps.append(d)
        if force or not _fresh(o, d):
            jobs.append(([nvcc] + flags + ["-c", s, "-o", o], o, d))
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            list(ex.map(lambda j: _run(j[0]), jobs))
        for _, o, d in jobs:
            _stamp(o, d)
    lib_digest = hashlib.sha256("".join(stamps).encode()).hexdigest()
    if force or jobs or not _fresh(LIB, lib_digest):
        # extern "C" entry points are exported explicitly; everything else stays hidden
        _run([nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                      "-Xcompiler", "-fPIC"])
        _stamp(LIB, lib_digest)
    return LIB


def lib_is_current() -> bool:
    """True when libfp8_b200.so was built from exactly the sources and flags in the tree (no compiler needed)."""
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.join(ROOT, "include", "fp8_b200.h")]
    flags = NVCC_FLAGS + EXTRA_NVCC_FLAGS
    stamps = [_digest([os.path.join(CSRC, src)] + hdrs, flags) for src in CU_SOURCES]
    return _fresh(LIB, hashlib.sha256("".join(stamps).encode()).hexdigest())


def build_ext(force: bool = False) -> str:
    import torch
    from torch.utils import cpp_extension as ce

    target = ext_path()
    src = os.path.join(CSRC, "fp8_bridge.cpp")
    digest = _digest([src, os.path.join(ROOT, "include", "fp8_b200.h")], [torch.__version__, sysconfig.get_config_var("EXT_SUFFIX")])
    if not force and _fresh(target, digest):
        return target
    inc = ce.include_paths() + [sysconfig.get_paths()["include"], "/usr/local/cuda/include"]
    tlib = os.path.join(os.path.dirname(torch.__file__), "lib")
    cxx = os.environ.get("CXX", "g++")
    cmd = [cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden",
           "-DTORCH_EXTENSION_NAME=fp8_metal", "-DTORCH_API_INCLUDE_EXTENSION_H",
           f"-D_GLIBCXX_USE_CXX11_ABI={int(torch._C._GLIBCXX_USE_CXX11_ABI)}", "-Wno-attributes"]
    for i in inc:
        cmd += ["-isystem", i]
    cmd += [src, "-o", target, f"-L{HERE}", "-l:libfp8_b200.so", "-Wl,-rpath,$ORIGIN",
            f"-L{tlib}", "-ltorch", "-ltorch_cpu", "-ltorch_python", "-lc10", "-lc10_cuda", "-ltorch_cuda"]
    _run(cmd)
    _stamp(target, digest)
    return target


def build_all(force: bool = False, ext: bool = True):
    out = [build_lib(force)]
    if ext and not PROFILE:
        out.append(build_ext(force))
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--no-ext", action="store_true")
    a = ap.parse_args()
    for p in build_all(a.force, not a.no_ext):
        print("built", os.path.relpath(p, ROOT))
    sys.exit(0)
