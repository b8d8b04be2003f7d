"""ctypes bindings to the closest-point CHECKERS (test infrastructure only):

  tests/point_query/liboracle_point.so  oracle_closest_point: the contract of b2rt_closest_point (include/b2rt.h) by brute
                                        force over the CLTriangle array, threaded; independent of the product's sources
                                        (tests/point_query/oracle_point.c)
  tests/point_query/libemu_point.so     tests/emu/emu.cpp plus the product's closest-point walk (csrc/point_query.cuh) on
                                        the host, and a direct check of its culling lemma (tests/point_query/emu_point.cpp)

The emulation library carries its own copy of the emulated scene: call emu_build() of THIS module before the emu_* calls.
Nothing here is reachable from the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "point_query")
ORACLE_SRC = [os.path.join(DIR, "oracle_point.c")]
EMU_SRC = [os.path.join(DIR, "emu_point.cpp"), os.path.join(ol.EMU_DIR, "emu.cpp"), os.path.join(ol.EMU_DIR, "warp_emu.cpp")] + \
          [os.path.join(ol.CSRC, f) for f in ("point_query.cuh", "traverse.cuh", "coop.cuh", "wide_bvh.cpp", "wide_bvh.h", "b2rt_types.h")]
QUERY = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("max_d2", "<f4")])
PHIT = np.dtype([("d2", "<f4"), ("u", "<f4"), ("v", "<f4"), ("tri", "<u4")])
_cache = {}


def build_oracle_point():
    out = os.path.join(DIR, "liboracle_point.so")
    if ol._stale(out, ORACLE_SRC):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                               ORACLE_SRC[0], "-o", out, "-lm"])
    return out


def build_emu_point():
    out = os.path.join(DIR, "libemu_point.so")
    if ol._stale(out, EMU_SRC):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-frounding-math",
                               "-fno-fast-math", "-pthread", "-x", "c++", "-I", ol.CSRC, EMU_SRC[0],
                               os.path.join(ol.EMU_DIR, "warp_emu.cpp"), os.path.join(ol.CSRC, "wide_bvh.cpp"), "-o", out])
    return out


def build_all():
    return build_oracle_point(), build_emu_point()


def _oracle():
    if "oracle" not in _cache:
        L = C.CDLL(build_oracle_point())
        L.oracle_closest_point.restype = None
        L.oracle_closest_point.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int]
        L.oracle_closest_on_triangle.restype = None
        L.oracle_closest_on_triangle.argtypes = [C.c_void_p] * 5
        _cache["oracle"] = L
    return _cache["oracle"]


def _emu():
    if "emu" not in _cache:
        L = C.CDLL(build_emu_point())
        L.emu_build.restype = C.c_char_p
        L.emu_build.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(ol.EmuStats)]
        L.emu_closest_point.restype = None
        L.emu_closest_point.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(ol.EmuStats)]
        L.emu_point_lb_check.restype = None
        L.emu_point_lb_check.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.emu_closest_on_triangle.restype = None
        L.emu_closest_on_triangle.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        _cache["emu"] = L
    return _cache["emu"]


def queries(points, max_d2=np.inf):
    """Pack (n, 3) points and a scalar or (n,) max_d2 into b2rt_point_query records."""
    p = np.asarray(points, dtype=np.float32).reshape(-1, 3)
    q = np.empty(p.shape[0], dtype=QUERY)
    q["x"], q["y"], q["z"] = p[:, 0], p[:, 1], p[:, 2]
    q["max_d2"] = max_d2
    return q


def oracle_closest_point(tris, q, threads=0):
    q = np.ascontiguousarray(q, dtype=QUERY)
    out = np.empty(q.shape[0], dtype=PHIT)
    _oracle().oracle_closest_point(ol._p(tris), tris.shape[0], ol._p(q), q.shape[0], ol._p(out), threads)
    return out


def oracle_on_triangle(p, a, b, c):
    """(d2, u, v) of the oracle's distance routine for one point and one triangle."""
    arr = [np.ascontiguousarray(np.asarray(x, dtype=np.float32)[:3]) for x in (p, a, b, c)]
    out = np.zeros(3, dtype=np.float32)
    _oracle().oracle_closest_on_triangle(*[ol._p(x) for x in arr], ol._p(out))
    return out


def emu_on_triangles(points, abc):
    """(n, 3) of (d2, u, v) from the product's closest_on_triangle for points (n, 3) and triangles (n, 3, 3)."""
    p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    t = np.ascontiguousarray(abc, dtype=np.float32).reshape(-1, 9)
    out = np.empty((p.shape[0], 3), dtype=np.float32)
    _emu().emu_closest_on_triangle(ol._p(p), ol._p(t), p.shape[0], ol._p(out))
    return out


def emu_build(tris, nodes):
    st = ol.EmuStats()
    err = _emu().emu_build(ol._p(nodes), nodes.shape[0], ol._p(tris), tris.shape[0], C.byref(st))
    if err:
        raise RuntimeError(err.decode())
    return st


def emu_closest_point(q, stats=None):
    """The product's wide walk (point_query.cuh) on the host over the scene of the last emu_build()."""
    q = np.ascontiguousarray(q, dtype=QUERY)
    st = stats if stats is not None else ol.EmuStats()
    out = np.empty(q.shape[0], dtype=PHIT)
    _emu().emu_closest_point(ol._p(q), q.shape[0], ol._p(out), C.byref(st))
    return out


def emu_lb_check(q):
    """(violations, children checked): children of the emulated tree whose lb exceeds the smallest d2 below them."""
    q = np.ascontiguousarray(q, dtype=QUERY)
    v, c = C.c_uint64(0), C.c_uint64(0)
    _emu().emu_point_lb_check(ol._p(q), q.shape[0], C.byref(v), C.byref(c))
    return int(v.value), int(c.value)
