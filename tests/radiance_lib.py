"""ctypes bindings to the radiance CHECKER (test infrastructure only):

  tests/radiance/liboracle_radiance.so  the contract of b2rt_trace_radiance (include/b2rt.h): the oracle's path loop with
                                        the ray's tmax on segment 0, over the kernels' powf / sinf / cosf
                                        (tests/radiance/oracle_radiance.c, which includes tests/frame_oracle/oracle_devlibm.c
                                        and through it oracle/rt_oracle.c unchanged)

Nothing here is reachable from the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

import frame_oracle_lib as fl
import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "radiance")
SRC = [os.path.join(DIR, "oracle_radiance.c")] + fl.ORACLE_SRC
RADIANCE = np.dtype([("r", "<f4"), ("g", "<f4"), ("b", "<f4"), ("seed", "<u4")])
_cache = {}


def build_oracle_radiance():
    out = os.path.join(DIR, "liboracle_radiance.so")
    if ol._stale(out, SRC):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                               "-Wno-unused-function", SRC[0], "-o", out, "-lm"])
    return out


def _lib():
    if "lib" not in _cache:
        L = C.CDLL(build_oracle_radiance())
        vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32
        L.oracle_radiance.argtypes = [vp, vp, vp, u32, vp, vp, u64, i32, i32, C.c_float, vp, C.c_int]
        L.oracle_radiance.restype = None
        L.oracle_render_path.argtypes = [vp, vp, vp, vp, vp, u64, i32, i32, C.c_float, vp, C.c_int]
        L.oracle_render_path.restype = None
        _cache["lib"] = L
    return _cache["lib"]


def _args(tris, nodes, mats, rays, seeds):
    rays = np.ascontiguousarray(rays)
    seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
    assert seeds.shape == (rays.shape[0],)
    mats = np.ascontiguousarray(mats)
    return rays, seeds, mats, np.empty(rays.shape[0], dtype=RADIANCE)


def oracle_radiance(tris, nodes, mats, rays, seeds, bounces, light_type=0, sky=1.0, threads=0):
    """The records b2rt_trace_radiance must return for these rays and seeds."""
    rays, seeds, mats, out = _args(tris, nodes, mats, rays, seeds)
    _lib().oracle_radiance(ol._p(tris), ol._p(nodes), ol._p(mats), mats.nbytes // 64, ol._p(rays), ol._p(seeds), rays.shape[0],
                           int(bounces), int(light_type), float(sky), ol._p(out), threads)
    return out


def oracle_render_path(tris, nodes, mats, rays, seeds, bounces, light_type=0, sky=1.0, threads=0):
    """The oracle's own render_path (100000 on every segment) from the same rays and seeds."""
    rays, seeds, mats, out = _args(tris, nodes, mats, rays, seeds)
    _lib().oracle_render_path(ol._p(tris), ol._p(nodes), ol._p(mats), ol._p(rays), ol._p(seeds), rays.shape[0], int(bounces),
                              int(light_type), float(sky), ol._p(out), threads)
    return out


def same(got, want):
    """Bit for bit, except that NaN channels compare equal whatever their payload (the CPU's default NaN differs from the
    GPU's)."""
    g = np.ascontiguousarray(got).view(np.uint32).reshape(-1, 4)
    w = np.ascontiguousarray(want).view(np.uint32).reshape(-1, 4)
    gf, wf = g[:, :3].view(np.float32), w[:, :3].view(np.float32)
    ok = (g == w).all(axis=1) | (((g[:, :3] == w[:, :3]) | (np.isnan(gf) & np.isnan(wf))).all(axis=1) & (g[:, 3] == w[:, 3]))
    bad = np.flatnonzero(~ok)
    assert bad.size == 0, "%d of %d records differ, first %s: got %s want %s" % (
        bad.size, ok.size, bad[:5], np.asarray(got)[bad[:3]], np.asarray(want)[bad[:3]])
