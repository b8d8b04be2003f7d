"""The frame-path checkers (test infrastructure only):

  tests/frame_oracle/liboracle_devlibm.so  the oracle (oracle/rt_oracle.c, included as it stands) with powf / sinf / cosf
                                           evaluated like the frame kernels' pow_cr / sin_cr / cos_cr: fp64, rounded once
                                                                                      (tests/frame_oracle/oracle_devlibm.c)
  tests/frame_oracle/libshadeprobe.so      the kernels' shading functions (csrc/shade.cuh) on the device, one record per
                                           thread                                      (tests/frame_oracle/shade_probe.cu)

Both run the same 16-word records (OP_* below), so a record's outputs compare bit for bit. oracle_render() has the
signature of oracle_lib.oracle_render. Nothing here is reachable from the product package.
"""
import ctypes as C
import importlib.util
import os
import subprocess

import numpy as np

import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "frame_oracle")
PKG = os.path.join(ol.ROOT, "mini-opencl-raytracer_b200")
ORACLE_SRC = [os.path.join(DIR, "oracle_devlibm.c"), os.path.join(ol.ORACLE_DIR, "rt_oracle.c"), os.path.join(ol.ORACLE_DIR, "rt_oracle.h")]
PROBE_SRC = [os.path.join(DIR, "shade_probe.cu"), os.path.join(PKG, "build.py")] + \
            [os.path.join(ol.CSRC, f) for f in ("shade.cuh", "traverse.cuh", "b2rt_types.h")]

OP_POW, OP_SINCOS, OP_FRAME, OP_BRDF, OP_LIGHT, OP_CAMERA, OP_RND, OP_ACCUMULATE = range(8)
_cache = {}


def build_oracle_devlibm():
    out = os.path.join(DIR, "liboracle_devlibm.so")
    if ol._stale(out, ORACLE_SRC):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                               "-Wno-unused-function", ORACLE_SRC[0], "-o", out, "-lm"])
    return out


def build_shade_probe():
    """nvcc with the product's flags (build.NVCC_FLAGS: sm_100a, -fmad=false, IEEE division and square root)."""
    out = os.path.join(DIR, "libshadeprobe.so")
    if ol._stale(out, PROBE_SRC):
        spec = importlib.util.spec_from_file_location("b2rt_build", os.path.join(PKG, "build.py"))
        build = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(build)
        subprocess.check_call([build.NVCC] + build.NVCC_FLAGS + ["-shared", PROBE_SRC[0], "-o", out])
    return out


def _oracle():
    if "oracle" not in _cache:
        L = C.CDLL(build_oracle_devlibm())
        vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
        L.oracle_render.argtypes = [vp, vp, vp, vp, u32, u32, u32, i32, i32, C.c_float, vp, vp, vp, u64, u64, C.c_int]
        L.oracle_render.restype = None
        L.fo_run.argtypes = [C.c_int, u64, vp, vp]
        L.fo_run.restype = None
        L.fo_camera_angle.restype = C.c_float
        _cache["oracle"] = L
    return _cache["oracle"]


def _probe():
    if "probe" not in _cache:
        L = C.CDLL(build_shade_probe())
        L.shade_probe_run.argtypes = [C.c_int, C.c_uint64, C.c_void_p, C.c_void_p]
        L.shade_probe_run.restype = C.c_int
        _cache["probe"] = L
    return _cache["probe"]


def records(n):
    """n zeroed input records (uint32 (n, 16)); write floats through .view(np.float32)."""
    return np.zeros((n, 16), dtype=np.uint32)


def oracle_run(op, rec):
    rec = np.ascontiguousarray(rec, dtype=np.uint32)
    out = np.empty_like(rec)
    _oracle().fo_run(op, rec.shape[0], ol._p(rec), ol._p(out))
    return out


def probe_run(op, rec):
    rec = np.ascontiguousarray(rec, dtype=np.uint32)
    out = np.empty_like(rec)
    err = _probe().shade_probe_run(op, rec.shape[0], ol._p(rec), ol._p(out))
    if err:
        raise RuntimeError("shade probe: CUDA error %d" % err)
    return out


def camera_angle():
    return float(_oracle().fo_camera_angle())


def oracle_render(tris, nodes, mats, result, width, height, frame_count, bounces, light_type=0, sky=1.0,
                  pos=(0.0, -25.0, 8.5), front=(0.0, 1.0, 0.0), up=(0.0, 0.0, 1.0), gid0=0, gid1=None, threads=0):
    gid1 = width * height if gid1 is None else gid1
    a, b, c = ol._v3(pos), ol._v3(front), ol._v3(up)
    _oracle().oracle_render(ol._p(tris), ol._p(nodes), ol._p(mats), ol._p(result), width, height, frame_count, bounces,
                            light_type, sky, ol._p(a), ol._p(b), ol._p(c), gid0, gid1, threads)
    return result
