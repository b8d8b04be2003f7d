#!/usr/bin/env python3
"""In-tree build of the product libraries (no CPU fallback is produced):

  csrc/  -> libb2rt.so      C ABI of include/b2rt.h + the sm_100a kernels (nvcc)
  host/  -> libglaze3d.so   headless C++ mirror of the reference's host classes
                            (CLRaytracer / CLEngineBase / CLBVHScene / CLOBJloader ...),
                            linked against libb2rt.so

nvcc cross-compiles sm_100a without a GPU, so this runs in the CPU container;
the built .so files are git-ignored but travel to the GPU box with gpurun.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
INCLUDE = os.path.join(ROOT, "include")
LIB_B2RT = os.path.join(HERE, "libb2rt.so")
LIB_HOST = os.path.join(HERE, "libglaze3d.so")
SCENEGEN = os.path.join(HERE, "scenegen")        # stand-alone synthetic-scene writer (host/scene_gen.cpp with its main)

NVCC = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-fmad=false", "-diag-suppress", "549", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
              "-Xcompiler", "-fPIC,-ffp-contract=off,-Wall", "-I", INCLUDE, "-I", CSRC]
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-I", INCLUDE, "-I", HOST]


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print("[build]", " ".join(cmd), flush=True)
    subprocess.check_call(cmd)


def build_b2rt(force=False, verbose=True):
    srcs = [os.path.join(CSRC, f) for f in ("kernels.cu", "lbvh.cu", "api.cu", "multi.cu", "refit.cu", "scene_build.cu", "wide_bvh.cpp")]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "b2rt.h"), __file__]
    if not force and not _stale(LIB_B2RT, deps):
        return LIB_B2RT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s) + ".o")
        _run([NVCC] + NVCC_FLAGS + ["-x", "cu", "-c", s, "-o", o], verbose)
        objs.append(o)
    _run([NVCC, "-shared", "-o", LIB_B2RT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-ldl"], verbose)
    return LIB_B2RT


def build_host(force=False, verbose=True):
    if not os.path.isdir(HOST):
        return None
    srcs = [os.path.join(HOST, f) for f in sorted(os.listdir(HOST)) if f.endswith(".cpp")]
    deps = srcs + [os.path.join(HOST, f) for f in os.listdir(HOST)] + [os.path.join(INCLUDE, "b2rt.h"), LIB_B2RT, __file__]
    if not force and not _stale(LIB_HOST, deps):
        return LIB_HOST
    cmd = ["g++"] + CXX_FLAGS + ["-shared", "-o", LIB_HOST] + srcs + ["-L", HERE, "-lb2rt", "-Wl,-rpath,$ORIGIN", "-pthread"]
    _run(cmd, verbose)
    return LIB_HOST


def build_scenegen(force=False, verbose=True):
    src = os.path.join(HOST, "scene_gen.cpp")
    if force or _stale(SCENEGEN, [src, __file__]):
        _run(["g++", "-std=c++17", "-O2", "-DB2RT_SCENEGEN_MAIN", src, "-o", SCENEGEN], verbose)
    return SCENEGEN


def build_all(force=False, verbose=True):
    out = build_b2rt(force, verbose), build_host(force, verbose)
    build_scenegen(force, verbose)
    return out


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv))
