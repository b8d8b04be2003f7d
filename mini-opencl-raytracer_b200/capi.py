"""ctypes view of libb2rt.so (include/b2rt.h). No compute happens in Python and there is
no fallback: a missing library or CUDA device raises."""
import ctypes as C
import os
import time

import numpy as np

from .layouts import HIT_DTYPE, MAT_BYTES, NODE_BYTES, POINT_HIT_DTYPE, POINT_QUERY_DTYPE, RADIANCE_DTYPE, RAY_DTYPE, TRI_BYTES

MISS = 0xFFFFFFFF
HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ARG_BUFFER_OUT, ARG_BUFFER_SCENE, ARG_BUFFER_NODE, ARG_BUFFER_MATERIAL = 0, 1, 2, 3
ARG_WIDTH, ARG_HEIGHT, ARG_FRAME_COUNT, ARG_FRAME_SEED = 4, 5, 6, 7
ARG_LIGHT_BOUNCES, ARG_LIGHT_TYPE, ARG_SKYBOX_INTENSITY = 8, 9, 10
ARG_CAMERA_POS, ARG_CAMERA_FRONT, ARG_CAMERA_UP = 11, 12, 13
OPT_TRAVERSAL, OPT_COUNTERS, OPT_BLOCKS_PER_SM, OPT_RENDER_MODE, OPT_REFILL_MIN, OPT_LEAF_BIAS, OPT_WAVEFRONT_LANES, OPT_COOP_MAX, OPT_L2_PERSIST, OPT_STAGE_TIMES, OPT_WAVEFRONT_GRID_SPLIT, OPT_RESUME_MAX, OPT_TAIL_HELP, OPT_SHARD_FENCE = 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13
MEM_WRITE_ONLY, MEM_READ_ONLY, MEM_COPY_HOST_PTR = 1 << 1, 1 << 2, 1 << 5

# every symbol include/b2rt.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "b2rt_create", "b2rt_destroy", "b2rt_last_error", "b2rt_status_string", "b2rt_buffer_create",
    "b2rt_buffer_release", "b2rt_set_arg", "b2rt_execute", "b2rt_execute_range", "b2rt_execute_bands", "b2rt_read_buffer",
    "b2rt_finish", "b2rt_host_register", "b2rt_host_unregister", "b2rt_upload_scene", "b2rt_resize", "b2rt_read_pixels", "b2rt_read_pixels_rgba8", "b2rt_trace_closest",
    "b2rt_trace_any", "b2rt_build_bvh", "b2rt_trace_closest_device", "b2rt_trace_any_device", "b2rt_camera_rays_device",
    "b2rt_device_pointer", "b2rt_bound_buffer", "b2rt_scene_info_get", "b2rt_set_option",
    "b2rt_get_counters", "b2rt_reset_counters", "b2rt_launch_count", "b2rt_device_count",
    "b2rt_create_multi", "b2rt_group_size", "b2rt_group_info", "b2rt_comm_unique_id", "b2rt_comm_init", "b2rt_comm_share_output",
    "b2rt_execute_shard", "b2rt_shard_bands", "b2rt_refit_scene", "b2rt_stage_times",
    "b2rt_build_scene_device", "b2rt_refit_scene_device", "b2rt_trace_multi", "b2rt_trace_multi_device",
    "b2rt_closest_point", "b2rt_closest_point_device", "b2rt_trace_radiance", "b2rt_trace_radiance_device",
]
MULTI_MAX_HITS = 64          # B2RT_MULTI_MAX_HITS: largest k of b2rt_trace_multi
# status bits of b2rt_refit_scene_device
REFIT_NONFINITE, REFIT_DUPLICATE, REFIT_RANGE, REFIT_LEAF_BOX, REFIT_ORDER = 1, 2, 4, 8, 16


class SceneInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_triangles", "n_nodes", "n_materials", "n_wide_nodes", "n_leaf_blocks",
                                          "wide_node_bytes", "leaf_bytes", "shading_bytes")] + \
               [(n, C.c_uint32) for n in ("max_depth_binary", "max_depth_wide", "sm_count", "reserved")]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "wide_nodes", "leaf_blocks", "leaf_gate_pass", "tri_tests",
                                          "bytes_fetched", "node_phases", "node_phase_lanes", "leaf_phases",
                                          "leaf_phase_lanes", "refills", "refill_lanes", "max_steps_per_ray",
                                          "stack_overflows", "coop_rays", "coop_steps", "coop_max_steps", "coop_max_rounds", "resumed_rays")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class B2RTError(RuntimeError):
    def __init__(self, status, text):
        super().__init__("b2rt status %d (%s): %s" % (status, _status_name(status), text))
        self.status = status


def lib_path():
    # B2RT_LIB: developer override to A/B another build of the same library
    return os.environ.get("B2RT_LIB") or os.path.join(HERE, "libb2rt.so")


def lib():
    """Load libb2rt.so. Fails loudly when it has not been built (no fallback exists)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError("%s is missing: run `python mini-opencl-raytracer_b200/build.py` "
                          "(there is no CPU or PyTorch fallback for the traversal kernels)" % p)
    L = C.CDLL(p, mode=C.RTLD_GLOBAL)
    vp, u64, u32, sz = C.c_void_p, C.c_uint64, C.c_uint32, C.c_size_t
    sig = {
        "b2rt_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "b2rt_destroy": (None, [vp]),
        "b2rt_last_error": (C.c_char_p, [vp]),
        "b2rt_status_string": (C.c_char_p, [C.c_int]),
        "b2rt_buffer_create": (C.c_int, [vp, u32, sz, vp, C.POINTER(u64)]),
        "b2rt_buffer_release": (C.c_int, [vp, u64]),
        "b2rt_set_arg": (C.c_int, [vp, u32, vp, sz]),
        "b2rt_execute": (C.c_int, [vp, sz]),
        "b2rt_execute_range": (C.c_int, [vp, sz, sz]),
        "b2rt_execute_bands": (C.c_int, [vp, sz, C.c_uint32, C.c_uint32, C.c_uint32]),
        "b2rt_read_buffer": (C.c_int, [vp, u64, vp, sz]),
        "b2rt_finish": (C.c_int, [vp]),
        "b2rt_host_register": (C.c_int, [vp, vp, sz]),
        "b2rt_host_unregister": (C.c_int, [vp, vp]),
        "b2rt_upload_scene": (C.c_int, [vp, vp, u64, vp, u64, vp, u64]),
        "b2rt_build_bvh": (C.c_int, [vp, vp, u64, vp, u64, C.POINTER(u64), vp]),
        "b2rt_resize": (C.c_int, [vp, u32, u32]),
        "b2rt_read_pixels": (C.c_int, [vp, vp, sz]),
        "b2rt_read_pixels_rgba8": (C.c_int, [vp, vp, sz]),
        "b2rt_trace_closest": (C.c_int, [vp, vp, u64, vp]),
        "b2rt_trace_any": (C.c_int, [vp, vp, u64, vp]),
        "b2rt_trace_closest_device": (C.c_int, [vp, vp, u64, vp, vp]),
        "b2rt_trace_any_device": (C.c_int, [vp, vp, u64, vp, vp]),
        "b2rt_trace_multi": (C.c_int, [vp, vp, u64, u32, vp]),
        "b2rt_trace_multi_device": (C.c_int, [vp, vp, u64, u32, vp, vp]),
        "b2rt_closest_point": (C.c_int, [vp, vp, u64, vp]),
        "b2rt_closest_point_device": (C.c_int, [vp, vp, u64, vp, vp]),
        "b2rt_trace_radiance": (C.c_int, [vp, vp, vp, u64, vp]),
        "b2rt_trace_radiance_device": (C.c_int, [vp, vp, vp, u64, vp, vp]),
        "b2rt_camera_rays_device": (C.c_int, [vp, sz, sz, vp, vp]),
        "b2rt_device_pointer": (C.c_int, [vp, u64, C.POINTER(vp), C.POINTER(sz)]),
        "b2rt_bound_buffer": (C.c_int, [vp, u32, C.POINTER(u64)]),
        "b2rt_scene_info_get": (C.c_int, [vp, C.POINTER(SceneInfo)]),
        "b2rt_set_option": (C.c_int, [vp, u32, C.c_int64]),
        "b2rt_get_counters": (C.c_int, [vp, C.POINTER(Counters)]),
        "b2rt_reset_counters": (C.c_int, [vp]),
        "b2rt_launch_count": (u64, [vp]),
        "b2rt_device_count": (C.c_int, []),
        "b2rt_refit_scene": (C.c_int, [vp, vp, u64]),
        "b2rt_build_scene_device": (C.c_int, [vp, vp, u64, vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), vp]),
        "b2rt_refit_scene_device": (C.c_int, [vp, vp, u64, vp, vp, vp]),
        "b2rt_stage_times": (C.c_int, [vp, C.POINTER(u32), C.POINTER(C.c_float), u32, C.POINTER(u32)]),
        "b2rt_create_multi": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]),
        "b2rt_group_size": (C.c_int, [vp]),
        "b2rt_group_info": (C.c_int, [vp, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
        "b2rt_comm_unique_id": (C.c_int, [vp, sz]),
        "b2rt_comm_init": (C.c_int, [vp, vp, sz, C.c_int, C.c_int]),
        "b2rt_comm_share_output": (C.c_int, [vp]),
        "b2rt_execute_shard": (C.c_int, [vp]),
        "b2rt_shard_bands": (C.c_int, [u32, u32, C.c_int, C.c_int, C.POINTER(u64), C.POINTER(u32), C.POINTER(u32), C.POINTER(u32),
                                       C.POINTER(u64), C.POINTER(u64)]),
    }
    for name, (res, args) in sig.items():
        if not hasattr(L, name) and os.environ.get("B2RT_LIB"):
            continue                          # an older build of the library under A/B: newer entry points are simply absent
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _LIB = L
    return L


def _status_name(status):
    try:
        return lib().b2rt_status_string(status).decode()
    except Exception:  # noqa: BLE001
        return "?"


def device_count():
    return int(lib().b2rt_device_count())


def comm_unique_id():
    """128 bytes identifying a new NCCL communicator (b2rt_comm_unique_id); hand them to every rank's Context.comm_init."""
    buf = C.create_string_buffer(128)
    st = lib().b2rt_comm_unique_id(buf, 128)
    if st:
        raise B2RTError(st, lib().b2rt_last_error(None).decode())
    return buf.raw


def shard_bands(width, height, rank, world):
    """b2rt_shard_bands: (gid_begin, band_pixels, stride_pixels, n_full_bands, tail_begin, tail_end) of `rank`."""
    g, t0, t1 = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    b, s, n = C.c_uint32(0), C.c_uint32(0), C.c_uint32(0)
    st = lib().b2rt_shard_bands(int(width), int(height), int(rank), int(world), C.byref(g), C.byref(b), C.byref(s), C.byref(n), C.byref(t0), C.byref(t1))
    if st:
        raise B2RTError(st, "bad shard arguments")
    return g.value, b.value, s.value, n.value, t0.value, t1.value


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if isinstance(a, np.ndarray) else C.c_void_p(int(a))


def _raw(a, itemsize, what):
    a = np.ascontiguousarray(a)
    if a.nbytes % itemsize:
        raise ValueError("%s: %d bytes is not a whole number of %d-byte records" % (what, a.nbytes, itemsize))
    return a, a.nbytes // itemsize


class Context:
    """b2rt_context: what the reference reaches through CLContext + CLKernel (CLutils.h:116-145)."""

    @classmethod
    def borrow(cls, handle, device=0):
        """Wrap a b2rt_context owned by someone else (e.g. the C++ CLContext of host.Engine)."""
        self = cls.__new__(cls)
        self._L = lib()
        self._h = C.c_void_p(handle)
        self._borrowed = True
        self.device = int(device)
        return self

    def __init__(self, device=0):
        """device: one CUDA device id, or a sequence of ids for ONE handle driving all of them (b2rt_create_multi)."""
        self._L = lib()
        self._borrowed = False
        h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            st = self._L.b2rt_create_multi(ids, len(device), C.byref(h))
            device = device[0] if device else 0
        else:
            st = self._L.b2rt_create(int(device), C.byref(h))
        if st:
            raise B2RTError(st, self._L.b2rt_last_error(None).decode())
        self._h = h
        self.device = int(device)

    # ---- multi-GPU ------------------------------------------------------------------------------
    def group_size(self):
        return int(self._L.b2rt_group_size(self._h))

    def group_info(self):
        a, b = C.c_int(0), C.c_int(0)
        self._ck(self._L.b2rt_group_info(self._h, C.byref(a), C.byref(b)))
        return {"peer_store": bool(a.value), "nccl_loaded": bool(b.value)}

    def comm_init(self, unique_id, rank, world):
        """unique_id: the bytes of comm_unique_id() made on one rank and distributed to all."""
        buf = C.create_string_buffer(bytes(unique_id), len(unique_id))
        self._ck(self._L.b2rt_comm_init(self._h, buf, len(unique_id), int(rank), int(world)))

    def comm_share_output(self):
        self._ck(self._L.b2rt_comm_share_output(self._h))

    def execute_shard(self):
        self._ck(self._L.b2rt_execute_shard(self._h))

    def close(self):
        if getattr(self, "_h", None):
            if not getattr(self, "_borrowed", False):
                self._L.b2rt_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, st):
        if st:
            raise B2RTError(st, self._L.b2rt_last_error(self._h).decode())

    # ---- scene / arguments -------------------------------------------------------------
    def upload_scene(self, tris, nodes, mats):
        t, nt = _raw(tris, TRI_BYTES, "triangles")
        n, nn = _raw(nodes, NODE_BYTES, "nodes")
        m, nm = _raw(mats, MAT_BYTES, "materials")
        self._ck(self._L.b2rt_upload_scene(self._h, _ptr(t), nt, _ptr(n), nn, _ptr(m), nm))

    def refit_scene(self, tris):
        """b2rt_refit_scene: new vertex data (same triangle count and order) for the bound scene."""
        tris, n = _raw(tris, 256, "CLTriangle")
        self._ck(self._L.b2rt_refit_scene(self._h, _ptr(tris), n))

    def read_nodes(self):
        """The bound CLLinearBVHNode buffer (slot 2) read back: (n, 48) uint8."""
        buf = C.c_uint64(0)
        self._ck(self._L.b2rt_bound_buffer(self._h, 2, C.byref(buf)))
        n = self.scene_info()["n_nodes"]
        out = np.empty((n, 48), dtype=np.uint8)
        self._ck(self._L.b2rt_read_buffer(self._h, buf, _ptr(out), out.nbytes))
        self.finish()
        return out

    def build_bvh(self, tris):
        """b2rt_build_bvh: binary BVH over loader-order triangles on the GPU, in the reference's format.
        Returns (re-ordered triangles, nodes, order) with order[k] = input index of output triangle k."""
        t, nt = _raw(tris, TRI_BYTES, "triangles")
        nodes = np.zeros((2 * nt - 1, NODE_BYTES), dtype=np.uint8)
        order = np.empty(nt, dtype=np.uint32)
        n_nodes = C.c_uint64(0)
        t0 = time.perf_counter()
        self._ck(self._L.b2rt_build_bvh(self._h, _ptr(t), nt, _ptr(nodes), nodes.shape[0], C.byref(n_nodes), _ptr(order)))
        self.last_build_seconds = time.perf_counter() - t0          # the C call alone (grouping, device build, flattening)
        return np.ascontiguousarray(t.reshape(nt, TRI_BYTES)[order]), nodes[: n_nodes.value].copy(), order

    def build_scene_device(self, d_triangles, n, d_order=0, stream=0):
        """b2rt_build_scene_device: the whole scene built on the device from n loader-order CLTriangles at device address
        d_triangles (e.g. a torch CUDA tensor's data_ptr()). Binds the two new buffers to slots 1 and 2; bind the
        materials first. d_order: optional device uint32[n] receiving order[k] = input index of triangle k.
        Returns (triangle buffer id, node buffer id, node count)."""
        bt, bn, nn = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        t0 = time.perf_counter()
        self._ck(self._L.b2rt_build_scene_device(self._h, C.c_void_p(int(d_triangles)), int(n), C.c_void_p(int(d_order)), C.byref(bt), C.byref(bn),
                                                 C.byref(nn), C.c_void_p(int(stream))))
        self.last_build_seconds = time.perf_counter() - t0
        return bt.value, bn.value, nn.value

    def refit_scene_device(self, d_triangles, n, d_status, d_order=0, stream=0):
        """b2rt_refit_scene_device: refit the bound scene from n CLTriangles at device address d_triangles -- scene order,
        or loader order gathered through d_order (the build's device order). d_status: device uint32 that receives the
        REFIT_* bits on the stream. Enqueued behind the work on `stream` (0 = the context's stream) and the context's
        stream; does not wait for the device on a single-device handle."""
        self._ck(self._L.b2rt_refit_scene_device(self._h, C.c_void_p(int(d_triangles)), int(n), C.c_void_p(int(d_order)),
                                                 C.c_void_p(int(d_status)), C.c_void_p(int(stream))))

    def read_scene(self):
        """The bound triangle (slot 1) and node (slot 2) buffers read back: ((n, 256) uint8, (m, 48) uint8)."""
        out = []
        for slot, rec in ((1, TRI_BYTES), (2, NODE_BYTES)):
            buf, size, ptr = C.c_uint64(0), C.c_size_t(0), C.c_void_p()
            self._ck(self._L.b2rt_bound_buffer(self._h, slot, C.byref(buf)))
            self._ck(self._L.b2rt_device_pointer(self._h, buf, C.byref(ptr), C.byref(size)))
            a = np.empty((size.value // rec, rec), dtype=np.uint8)
            self._ck(self._L.b2rt_read_buffer(self._h, buf, _ptr(a), a.nbytes))
            out.append(a)
        self.finish()
        return out[0], out[1]

    def set_materials(self, mats):
        """A new material buffer (CLMaterial[]) bound to slot 3; the previous one is released. Returns its id."""
        m, nm = _raw(mats, MAT_BYTES, "materials")
        old, buf = C.c_uint64(0), C.c_uint64(0)
        self._ck(self._L.b2rt_bound_buffer(self._h, 3, C.byref(old)))
        self._ck(self._L.b2rt_buffer_create(self._h, MEM_READ_ONLY | MEM_COPY_HOST_PTR, m.nbytes, _ptr(m), C.byref(buf)))
        self.set_arg(3, buf.value)
        if old.value and old.value != buf.value:
            self._ck(self._L.b2rt_buffer_release(self._h, old.value))
        return buf.value

    def resize(self, width, height):
        self._ck(self._L.b2rt_resize(self._h, int(width), int(height)))
        self.width, self.height = int(width), int(height)

    def set_arg(self, slot, value):
        v = np.ascontiguousarray(value)
        self._ck(self._L.b2rt_set_arg(self._h, int(slot), _ptr(v), v.nbytes))

    def set_frame(self, frame_count, bounces, light_type=0, sky=1.0, pos=(0.0, -25.0, 8.5), front=(0.0, 1.0, 0.0),
                  up=(0.0, 0.0, 1.0), seed=0):
        """The eight per-frame SetUniform calls of CLRaytracer::RenderFrame (CLRaytracer.cpp:36-47)."""
        L, h = self._L, self._h
        for slot, v in ((ARG_FRAME_COUNT, C.c_uint32(frame_count)), (ARG_FRAME_SEED, C.c_uint32(seed)), (ARG_LIGHT_BOUNCES, C.c_int32(bounces)),
                        (ARG_LIGHT_TYPE, C.c_int32(light_type)), (ARG_SKYBOX_INTENSITY, C.c_float(sky))):
            self._ck(L.b2rt_set_arg(h, slot, C.byref(v), 4))
        for slot, v in ((ARG_CAMERA_POS, pos), (ARG_CAMERA_FRONT, front), (ARG_CAMERA_UP, up)):
            f3 = (C.c_float * 4)(v[0], v[1], v[2], 0.0)
            self._ck(L.b2rt_set_arg(h, slot, f3, 16))

    def set_shading(self, bounces, light_type=0, sky=1.0):
        """Only the shading slots (light bounces, light type, sky intensity): all that trace_radiance needs besides the scene."""
        for slot, v in ((ARG_LIGHT_BOUNCES, C.c_int32(bounces)), (ARG_LIGHT_TYPE, C.c_int32(light_type)), (ARG_SKYBOX_INTENSITY, C.c_float(sky))):
            self._ck(self._L.b2rt_set_arg(self._h, slot, C.byref(v), 4))

    def set_option(self, option, value):
        self._ck(self._L.b2rt_set_option(self._h, int(option), int(value)))

    # ---- frame path -------------------------------------------------------------------------
    def execute(self, work_size):
        self._ck(self._L.b2rt_execute(self._h, int(work_size)))

    def execute_range(self, gid0, gid1):
        self._ck(self._L.b2rt_execute_range(self._h, int(gid0), int(gid1)))

    def execute_bands(self, gid0, band_pixels, stride_pixels, n_bands):
        """n_bands bands of band_pixels gids, band starts stride_pixels apart: one rank's share of a frame."""
        self._ck(self._L.b2rt_execute_bands(self._h, int(gid0), int(band_pixels), int(stride_pixels), int(n_bands)))

    def finish(self):
        self._ck(self._L.b2rt_finish(self._h))

    def host_register(self, array):
        self._ck(self._L.b2rt_host_register(self._h, _ptr(array), array.nbytes))

    def host_unregister(self, array):
        self._ck(self._L.b2rt_host_unregister(self._h, _ptr(array)))

    def read_pixels(self, out=None):
        n = self.width * self.height
        if out is None:
            out = np.empty((n, 4), dtype=np.float32)
        self._ck(self._L.b2rt_read_pixels(self._h, _ptr(out), out.nbytes))
        self.finish()
        return out

    def read_pixels_async(self, out):
        """b2rt_read_pixels without the finish: the copy is only enqueued (asynchronous for real when `out` is pinned,
        see host_register); the caller calls finish() before looking at `out`."""
        self._ck(self._L.b2rt_read_pixels(self._h, _ptr(out), out.nbytes))

    def read_pixels_rgba8(self, out=None):
        """Clamped 8-bit RGBA view of the accumulation image, quantised on the device (4 B/pixel read-back)."""
        n = self.width * self.height
        if out is None:
            out = np.empty((n, 4), dtype=np.uint8)
        self._ck(self._L.b2rt_read_pixels_rgba8(self._h, _ptr(out), out.nbytes))
        self.finish()
        return out

    def output_device_pointer(self):
        buf = C.c_uint64()
        self._ck(self._L.b2rt_bound_buffer(self._h, 0, C.byref(buf)))
        p, n = C.c_void_p(), C.c_size_t()
        self._ck(self._L.b2rt_device_pointer(self._h, buf.value, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    # ---- ray streams ------------------------------------------------------------------------
    def trace_closest(self, rays, hits=None):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        if hits is None:
            hits = np.empty(rays.shape[0], dtype=HIT_DTYPE)
        self._ck(self._L.b2rt_trace_closest(self._h, _ptr(rays), rays.shape[0], _ptr(hits)))
        return hits

    def trace_any(self, rays, occluded=None):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        if occluded is None:
            occluded = np.empty(rays.shape[0], dtype=np.uint32)
        self._ck(self._L.b2rt_trace_any(self._h, _ptr(rays), rays.shape[0], _ptr(occluded)))
        return occluded

    def trace_multi(self, rays, k):
        """The k nearest hits of every ray (b2rt_trace_multi): an (n, k) HIT_DTYPE array, each row sorted by t and
        padded with {tmax, 0, 0, MISS}."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.empty((rays.shape[0], max(int(k), 0)), dtype=HIT_DTYPE)
        self._ck(self._L.b2rt_trace_multi(self._h, _ptr(rays), rays.shape[0], int(k), _ptr(hits)))
        return hits

    def trace_multi_device(self, d_rays, n, k, d_hits, stream=0):
        """b2rt_trace_multi_device: d_hits holds n * k records of 16 bytes."""
        self._ck(self._L.b2rt_trace_multi_device(self._h, C.c_void_p(int(d_rays)), int(n), int(k), C.c_void_p(int(d_hits)),
                                                 C.c_void_p(int(stream))))

    def closest_point(self, queries):
        """The nearest surface point of the scene to every query (b2rt_closest_point): a POINT_HIT_DTYPE array of
        {d2, u, v, tri}; {max_d2, 0, 0, MISS} where no triangle lies within max_d2."""
        queries = np.ascontiguousarray(queries, dtype=POINT_QUERY_DTYPE)
        out = np.empty(queries.shape[0], dtype=POINT_HIT_DTYPE)
        self._ck(self._L.b2rt_closest_point(self._h, _ptr(queries), queries.shape[0], _ptr(out)))
        return out

    def closest_point_device(self, d_queries, n, d_out, stream=0):
        """b2rt_closest_point_device: n query and n result records of 16 bytes in device memory."""
        self._ck(self._L.b2rt_closest_point_device(self._h, C.c_void_p(int(d_queries)), int(n), C.c_void_p(int(d_out)),
                                                   C.c_void_p(int(stream))))

    def trace_radiance(self, rays, seeds):
        """The path-traced radiance of every ray (b2rt_trace_radiance): a RADIANCE_DTYPE array of {r, g, b, seed}, the
        seed being the RNG state after the path. Shading comes from the bound light bounces, light type, sky intensity and
        materials (set_shading or set_frame)."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        if seeds.shape != (rays.shape[0],):
            raise ValueError("one seed per ray: %d rays, seeds of shape %s" % (rays.shape[0], seeds.shape))
        out = np.empty(rays.shape[0], dtype=RADIANCE_DTYPE)
        self._ck(self._L.b2rt_trace_radiance(self._h, _ptr(rays), _ptr(seeds), rays.shape[0], _ptr(out)))
        return out

    def trace_radiance_device(self, d_rays, d_seeds, n, d_out, stream=0):
        """b2rt_trace_radiance_device: n rays (32 B), n uint32 seeds and n records of 16 bytes in device memory."""
        self._ck(self._L.b2rt_trace_radiance_device(self._h, C.c_void_p(int(d_rays)), C.c_void_p(int(d_seeds)), int(n),
                                                    C.c_void_p(int(d_out)), C.c_void_p(int(stream))))

    def trace_closest_device(self, d_rays, n, d_hits, stream=0):
        self._ck(self._L.b2rt_trace_closest_device(self._h, C.c_void_p(int(d_rays)), int(n), C.c_void_p(int(d_hits)),
                                                   C.c_void_p(int(stream))))

    def trace_any_device(self, d_rays, n, d_occ, stream=0):
        self._ck(self._L.b2rt_trace_any_device(self._h, C.c_void_p(int(d_rays)), int(n), C.c_void_p(int(d_occ)),
                                               C.c_void_p(int(stream))))

    def camera_rays_device(self, gid0, gid1, d_rays, stream=0):
        self._ck(self._L.b2rt_camera_rays_device(self._h, int(gid0), int(gid1), C.c_void_p(int(d_rays)),
                                                 C.c_void_p(int(stream))))

    # ---- introspection ------------------------------------------------------------------------
    def scene_info(self):
        s = SceneInfo()
        self._ck(self._L.b2rt_scene_info_get(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in SceneInfo._fields_}

    def stage_times(self):
        """[(stage name, ms)] of the last wavefront frame launch made with OPT_STAGE_TIMES = 1."""
        kinds, ms, n = (C.c_uint32 * 64)(), (C.c_float * 64)(), C.c_uint32(0)
        self._ck(self._L.b2rt_stage_times(self._h, kinds, ms, 64, C.byref(n)))
        names = {1: "generate", 2: "trace", 3: "tail", 4: "shade"}
        return [(names.get(kinds[i], "?"), float(ms[i])) for i in range(n.value)]

    def counters(self):
        c = Counters()
        self._ck(self._L.b2rt_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    def reset_counters(self):
        self._ck(self._L.b2rt_reset_counters(self._h))

    def launch_count(self):
        return int(self._L.b2rt_launch_count(self._h))
