"""ctypes view of libglaze3d.so: the C++ mirror of the reference's host classes (host/glaze3d.h).
Scene ingest (CLOBJloader + CLBVHScene build) runs on the CPU like in the reference; everything that
touches rays goes through libb2rt.so on the GPU."""
import ctypes as C
import os

import numpy as np

from . import capi
from .layouts import HIT_DTYPE, POINT_HIT_DTYPE, POINT_QUERY_DTYPE, RADIANCE_DTYPE, RAY_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class HostError(RuntimeError):
    def __init__(self, text, status=None):
        super().__init__(text)
        self.status = status                # the C++ CLException's code where the call reports it, else None


def lib_path():
    return os.path.join(HERE, "libglaze3d.so")


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    capi.lib()                      # libglaze3d.so links against libb2rt.so (rpath $ORIGIN)
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError("%s is missing: run `python mini-opencl-raytracer_b200/build.py`" % p)
    L = C.CDLL(p)
    vp, u64, cs, sz = C.c_void_p, C.c_uint64, C.c_char_p, C.c_size_t
    sig = {
        "g3d_scene_load": (vp, [cs, C.c_uint, cs, sz]),
        "g3d_scene_load_cached": (vp, [cs, C.c_uint, cs, C.POINTER(C.c_int), cs, sz]),
        "g3d_engine_load_scene_cached": (C.c_int, [vp, cs, C.c_uint, cs, C.POINTER(C.c_int), cs, sz]),
        "g3d_scene_load_triangles": (vp, [cs, cs, sz]),
        "g3d_engine_load_scene_device_bvh": (C.c_int, [vp, cs, cs, sz]),
        "g3d_engine_scene_from_device": (C.c_int, [vp, vp, C.c_uint64, vp, C.c_uint64, cs, sz]),
        "g3d_engine_scene_read_back": (C.c_int, [vp, cs, sz]),
        "g3d_engine_scene_refit_device": (C.c_int, [vp, vp, C.c_uint64, cs, sz]),
        "g3d_scene_from_triangles": (vp, [vp, u64, vp, u64, C.c_uint, cs, sz]),
        "g3d_scene_free": (None, [vp]),
        "g3d_scene_count": (u64, [vp, C.c_int]),
        "g3d_scene_data": (vp, [vp, C.c_int]),
        "g3d_engine_create": (vp, [C.c_int, C.c_int, C.c_int, cs, sz]),
        "g3d_engine_destroy": (None, [vp]),
        "g3d_engine_load_scene": (C.c_int, [vp, cs, C.c_uint, cs, sz]),
        "g3d_engine_adopt_scene": (C.c_int, [vp, vp, cs, sz]),
        "g3d_engine_set_camera": (None, [vp, vp, vp, vp]),
        "g3d_engine_set_render": (None, [vp, C.c_uint, C.c_int, C.c_int, C.c_float]),
        "g3d_engine_set_shard": (None, [vp, u64, u64]),
        "g3d_engine_render_frame": (C.c_int, [vp, cs, sz]),
        "g3d_engine_pixels": (vp, [vp]),
        "g3d_engine_set_display_readback": (None, [vp, C.c_int]),
        "g3d_engine_pixels8": (vp, [vp]),
        "g3d_engine_frame_count": (C.c_uint, [vp]),
        "g3d_engine_context": (vp, [vp]),
        "g3d_engine_scene": (vp, [vp]),
        "g3d_engine_trace_closest": (C.c_int, [vp, vp, u64, vp, cs, sz]),
        "g3d_engine_trace_any": (C.c_int, [vp, vp, u64, vp, cs, sz]),
        "g3d_engine_trace_multi": (C.c_int, [vp, vp, u64, C.c_uint32, vp, cs, sz]),
        "g3d_engine_closest_point": (C.c_int, [vp, vp, u64, vp, cs, sz]),
        "g3d_engine_trace_radiance": (C.c_int, [vp, vp, vp, u64, vp, cs, sz]),
        "g3d_write_icosphere_obj": (C.c_longlong, [cs, C.c_int, C.c_double, C.c_double, C.c_ulonglong]),
        "g3d_write_scattered_obj": (C.c_longlong, [cs, C.c_longlong, C.c_double, C.c_double, C.c_double, C.c_ulonglong]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _LIB = L
    return L


def _err():
    return C.create_string_buffer(512)


def _arrays(L, handle):
    out = []
    for which, size in ((0, 256), (1, 48), (2, 64)):
        n = int(L.g3d_scene_count(handle, which))
        if n:
            buf = (C.c_uint8 * (n * size)).from_address(L.g3d_scene_data(handle, which))
            out.append(np.frombuffer(buf, dtype=np.uint8).copy().reshape(n, size))
        else:
            out.append(np.zeros((0, size), dtype=np.uint8))
    return tuple(out)


def load_scene(obj_path, max_prims=4, cache=None):
    """CLOBJloader::Load + CLBVHScene build (no device): (tris, nodes, mats) as uint8 record arrays.
    cache: None = parse + build like the reference; True = binary scene cache beside the .obj; a path = that cache file.
    With a cache the return value gains a fourth element: whether the cache was hit."""
    L = lib()
    e = _err()
    if cache:
        hit = C.c_int(0)
        h = L.g3d_scene_load_cached(os.fsencode(obj_path), max_prims, None if cache is True else os.fsencode(cache), C.byref(hit), e, len(e))
        if not h:
            raise HostError(e.value.decode())
        try:
            return _arrays(L, h) + (bool(hit.value),)
        finally:
            L.g3d_scene_free(h)
    h = L.g3d_scene_load(os.fsencode(obj_path), max_prims, e, len(e))
    if not h:
        raise HostError(e.value.decode())
    try:
        return _arrays(L, h)
    finally:
        L.g3d_scene_free(h)


def load_triangles(obj_path):
    """CLOBJloader only: (tris, mats) in LOADER order, no BVH -- the input of Context.build_bvh / b2rt_build_bvh."""
    L = lib()
    e = _err()
    h = L.g3d_scene_load_triangles(os.fsencode(obj_path), e, len(e))
    if not h:
        raise HostError(e.value.decode())
    try:
        t, _, m = _arrays(L, h)
        return t, m
    finally:
        L.g3d_scene_free(h)


def build_scene(tris, mats, max_prims=4):
    """CLBVHScene build over caller-provided pre-loader triangles."""
    L = lib()
    e = _err()
    tris = np.ascontiguousarray(tris)
    mats = np.ascontiguousarray(mats)
    h = L.g3d_scene_from_triangles(tris.ctypes.data, tris.nbytes // 256, mats.ctypes.data, mats.nbytes // 64, max_prims, e, len(e))
    if not h:
        raise HostError(e.value.decode())
    try:
        return _arrays(L, h)
    finally:
        L.g3d_scene_free(h)


def write_icosphere_obj(path, frequency, radius=10.0, amplitude=0.08, seed=7):
    n = lib().g3d_write_icosphere_obj(os.fsencode(path), frequency, radius, amplitude, seed)
    if n < 0:
        raise HostError("could not write %s" % path)
    return int(n)


def write_scattered_obj(path, count, extent=50.0, edge_min=0.05, edge_max=0.5, seed=11):
    n = lib().g3d_write_scattered_obj(os.fsencode(path), count, extent, edge_min, edge_max, seed)
    if n < 0:
        raise HostError("could not write %s" % path)
    return int(n)


class Engine:
    """CLEngineBase + CLRaytracer on one GPU: Init, scene load, RenderFrame, ray streams."""

    def __init__(self, width, height, device=0):
        self._L = lib()
        e = _err()
        self._h = self._L.g3d_engine_create(device, width, height, e, len(e))
        if not self._h:
            raise HostError(e.value.decode())
        self.width, self.height, self.device = width, height, device

    def close(self):
        if getattr(self, "_h", None):
            self._L.g3d_engine_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc, e):
        if rc:
            raise HostError(e.value.decode())

    def load_scene(self, obj_path, max_prims=4, cache=None):
        """CLEngineBase.cpp:172-179 (new scene, Load, CreateBVHTrees + upload). cache as in host.load_scene; returns
        True when the binary scene cache was hit."""
        e = _err()
        if cache:
            hit = C.c_int(0)
            self._ck(self._L.g3d_engine_load_scene_cached(self._h, os.fsencode(obj_path), max_prims,
                                                          None if cache is True else os.fsencode(cache), C.byref(hit), e, len(e)), e)
            return bool(hit.value)
        self._ck(self._L.g3d_engine_load_scene(self._h, os.fsencode(obj_path), max_prims, e, len(e)), e)
        return False

    def load_scene_device_bvh(self, obj_path):
        """CLOBJloader::Load, then CLBVHScene::CreateBVHTreesDevice: the binary BVH is built on the GPU."""
        e = _err()
        self._ck(self._L.g3d_engine_load_scene_device_bvh(self._h, os.fsencode(obj_path), e, len(e)), e)

    def build_scene_device(self, d_triangles, n, mats):
        """A new scene from n loader-order CLTriangles at device address d_triangles (CLBVHScene::CreateBVHTreesFromDevice):
        built on the GPU, nothing read back; scene_arrays() is empty until read_back_scene()."""
        m = np.ascontiguousarray(mats)
        e = _err()
        self._ck(self._L.g3d_engine_scene_from_device(self._h, C.c_void_p(int(d_triangles)), int(n), m.ctypes.data, m.nbytes // 64, e, len(e)), e)

    def read_back_scene(self):
        """CLBVHScene::ReadBackScene: the device-built triangles and nodes into the host arrays."""
        e = _err()
        self._ck(self._L.g3d_engine_scene_read_back(self._h, e, len(e)), e)

    def refit_scene_device(self, d_triangles, n):
        """CLBVHScene::RefitFromDevice: new vertex data for the device scene from n CLTriangles at device address d_triangles,
        in loader order for a scene made by build_scene_device, else in scene order. Raises HostError (with .status) on
        failure, status -50 (CL_INVALID_ARG_VALUE) when the refit reported bad data."""
        e = _err()
        rc = self._L.g3d_engine_scene_refit_device(self._h, C.c_void_p(int(d_triangles)), int(n), e, len(e))
        if rc:
            raise HostError(e.value.decode(), rc)

    def scene_arrays(self):
        h = self._L.g3d_engine_scene(self._h)
        try:
            return _arrays(self._L, h)
        finally:
            self._L.g3d_scene_free(h)

    def set_camera(self, pos, front, up):
        a, b, c = (np.asarray(v, dtype=np.float32) for v in (pos, front, up))
        self._L.g3d_engine_set_camera(self._h, a.ctypes.data, b.ctypes.data, c.ctypes.data)

    def set_render(self, frame_count=1, bounces=9, light_type=0, sky=1.0):
        self._L.g3d_engine_set_render(self._h, frame_count, bounces, light_type, sky)

    def set_shard(self, gid0, gid1):
        self._L.g3d_engine_set_shard(self._h, gid0, gid1)

    def render_frame(self):
        """CLRaytracer::RenderFrame: 8 SetUniform, ExecuteKernel, ReadBuffer, Finish; ++m_FrameCount."""
        e = _err()
        self._ck(self._L.g3d_engine_render_frame(self._h, e, len(e)), e)

    def pixels(self):
        """View of CLRaytracer::pixels (W*H float3 = 4 floats each), valid until the engine is resized/closed."""
        buf = (C.c_float * (self.width * self.height * 4)).from_address(self._L.g3d_engine_pixels(self._h))
        return np.frombuffer(buf, dtype=np.float32).reshape(-1, 4)

    def set_display_readback(self, on=True):
        """RenderFrame reads back clamped 8-bit RGBA (pixels8) instead of the float image (pixels)."""
        self._L.g3d_engine_set_display_readback(self._h, 1 if on else 0)

    def pixels8(self):
        buf = (C.c_uint8 * (self.width * self.height * 4)).from_address(self._L.g3d_engine_pixels8(self._h))
        return np.frombuffer(buf, dtype=np.uint8).reshape(-1, 4)

    def context_handle(self):
        return self._L.g3d_engine_context(self._h)

    def trace_closest(self, rays, hits=None):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        if hits is None:
            hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        e = _err()
        self._ck(self._L.g3d_engine_trace_closest(self._h, rays.ctypes.data, rays.shape[0], hits.ctypes.data, e, len(e)), e)
        return hits

    def trace_any(self, rays, occluded=None):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        if occluded is None:
            occluded = np.empty(rays.shape[0], dtype=np.uint32)
        e = _err()
        self._ck(self._L.g3d_engine_trace_any(self._h, rays.ctypes.data, rays.shape[0], occluded.ctypes.data, e, len(e)), e)
        return occluded

    def trace_multi(self, rays, k):
        """CLRaytracer::TraceMulti: the k nearest hits of every ray as an (n, k) HIT_DTYPE array."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty((rays.shape[0], max(int(k), 0)), dtype=HIT_DTYPE)
        e = _err()
        self._ck(self._L.g3d_engine_trace_multi(self._h, rays.ctypes.data, rays.shape[0], int(k), hits.ctypes.data, e, len(e)), e)
        return hits

    def closest_point(self, queries):
        """CLRaytracer::ClosestPoint: the nearest surface point of the scene to every query as a POINT_HIT_DTYPE array."""
        queries = np.ascontiguousarray(queries, dtype=POINT_QUERY_DTYPE)
        out = np.empty(queries.shape[0], dtype=POINT_HIT_DTYPE)
        e = _err()
        self._ck(self._L.g3d_engine_closest_point(self._h, queries.ctypes.data, queries.shape[0], out.ctypes.data, e, len(e)), e)
        return out

    def trace_radiance(self, rays, seeds):
        """CLRaytracer::TraceRadiance: the path-traced radiance of every ray as a RADIANCE_DTYPE array {r, g, b, seed}."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        if seeds.shape != (rays.shape[0],):
            raise ValueError("one seed per ray: %d rays, seeds of shape %s" % (rays.shape[0], seeds.shape))
        out = np.empty(rays.shape[0], dtype=RADIANCE_DTYPE)
        e = _err()
        self._ck(self._L.g3d_engine_trace_radiance(self._h, rays.ctypes.data, seeds.ctypes.data, rays.shape[0], out.ctypes.data, e, len(e)), e)
        return out
