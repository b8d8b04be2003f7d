"""ctypes bindings to the multi-hit CHECKERS (test infrastructure only):

  tests/multi_hit/liboracle_multi.so  oracle_trace_multi: the oracle's reference walk (oracle/rt_oracle.c, included as it
                                      stands) keeping the k nearest hits                       (tests/multi_hit/oracle_multi.c)
  tests/multi_hit/libemu_multi.so     tests/emu/emu.cpp plus emu_trace_multi: the product's Lane with the HIT_MULTI policy
                                      (csrc/traverse.cuh) on the host, through trace_wide       (tests/multi_hit/emu_multi.cpp)

The emulation library carries its own copy of the emulated scene: call emu_build() of THIS module before emu_trace_multi().
Nothing here is reachable from the product package.
"""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle_lib as ol

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "multi_hit")
ORACLE_SRC = [os.path.join(DIR, "oracle_multi.c"), os.path.join(ol.ORACLE_DIR, "rt_oracle.c"), os.path.join(ol.ORACLE_DIR, "rt_oracle.h")]
EMU_SRC = [os.path.join(DIR, "emu_multi.cpp"), os.path.join(ol.EMU_DIR, "emu.cpp"), os.path.join(ol.EMU_DIR, "warp_emu.cpp")] + \
          [os.path.join(ol.CSRC, f) for f in ("traverse.cuh", "coop.cuh", "wide_bvh.cpp", "wide_bvh.h", "b2rt_types.h")]
_cache = {}


def build_oracle_multi():
    out = os.path.join(DIR, "liboracle_multi.so")
    if ol._stale(out, ORACLE_SRC):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                               "-Wno-unused-function", ORACLE_SRC[0], "-o", out, "-lm"])
    return out


def build_emu_multi():
    out = os.path.join(DIR, "libemu_multi.so")
    if ol._stale(out, EMU_SRC):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-frounding-math",
                               "-fno-fast-math", "-pthread", "-DB2_EMU_CHECK_CULLING", "-x", "c++", "-I", ol.CSRC, EMU_SRC[0],
                               os.path.join(ol.EMU_DIR, "warp_emu.cpp"), os.path.join(ol.CSRC, "wide_bvh.cpp"), "-o", out])
    return out


def build_all():
    return build_oracle_multi(), build_emu_multi()


def _oracle():
    if "oracle" not in _cache:
        L = C.CDLL(build_oracle_multi())
        L.oracle_trace_multi.restype = None
        L.oracle_trace_multi.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int]
        _cache["oracle"] = L
    return _cache["oracle"]


def _emu():
    if "emu" not in _cache:
        L = C.CDLL(build_emu_multi())
        L.emu_build.restype = C.c_char_p
        L.emu_build.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(ol.EmuStats)]
        L.emu_trace_multi.restype = None
        L.emu_trace_multi.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.POINTER(ol.EmuStats), C.c_uint32]
        L.emu_culling_violations.restype = C.c_uint64
        _cache["emu"] = L
    return _cache["emu"]


def oracle_trace_multi(tris, nodes, rays, k, threads=0):
    """The k nearest hits of every ray as an (n, k) HIT array (rows sorted by t, padded with {tmax, 0, 0, miss})."""
    rays = np.ascontiguousarray(rays)
    hits = np.empty((rays.shape[0], int(k)), dtype=ol.HIT)
    _oracle().oracle_trace_multi(ol._p(tris), ol._p(nodes), ol._p(rays), rays.shape[0], int(k), ol._p(hits), threads)
    return hits


def emu_build(tris, nodes):
    st = ol.EmuStats()
    err = _emu().emu_build(ol._p(nodes), nodes.shape[0], ol._p(tris), tris.shape[0], C.byref(st))
    if err:
        raise RuntimeError(err.decode())
    return st


def emu_trace_multi(rays, k, schedule=0, stats=None):
    """The product's HIT_MULTI walk on the host over the scene of the last emu_build(); schedule as for oracle_lib.emu_trace."""
    rays = np.ascontiguousarray(rays)
    st = stats if stats is not None else ol.EmuStats()
    hits = np.empty((rays.shape[0], int(k)), dtype=ol.HIT)
    _emu().emu_trace_multi(ol._p(rays), rays.shape[0], int(k), ol._p(hits), C.byref(st), schedule)
    return hits


def emu_culling_violations():
    """Children the exact node test lets through but the fast one culled, over every walk of this library (must stay 0)."""
    return int(_emu().emu_culling_violations())
