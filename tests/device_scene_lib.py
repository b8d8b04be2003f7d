"""Helpers for the device scene build tests: the scene-hooks library (tests/emu/scene_hooks.cu), which copies the compressed
wide BVH a handle derived back to the host, and loader-order triangles placed in device memory."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU_DIR = os.path.join(ROOT, "tests", "emu")
CSRC = os.path.join(ROOT, "mini-opencl-raytracer_b200", "csrc")
_cache = {}


def build_scene_hooks():
    """tests/emu/libscenehooks.so (nvcc, sm_100a); rebuilt when its source or the context layout changed."""
    out = os.path.join(EMU_DIR, "libscenehooks.so")
    src = os.path.join(EMU_DIR, "scene_hooks.cu")
    deps = [src, os.path.join(ROOT, "include", "b2rt.h")] + [os.path.join(CSRC, f) for f in ("context.h", "kernels.h", "b2rt_types.h")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC",
                               "-I", os.path.join(ROOT, "include"), "-I", CSRC, src, "-o", out])
    return out


def scene_hooks():
    if "hooks" not in _cache:
        L = C.CDLL(build_scene_hooks())
        L.b2rt_test_derived_arrays.restype = C.c_int
        L.b2rt_test_derived_arrays.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong)] + [C.c_void_p] * 5 + [C.POINTER(C.c_uint)]
        _cache["hooks"] = L
    return _cache["hooks"]


def derived_arrays(ctx):
    """What `ctx` (a product Context) derived: the five arrays as uint8, stack_bound and scene_info."""
    info = ctx.scene_info()                            # derives the scene where that is still pending
    L = scene_hooks()
    sizes = (C.c_ulonglong * 5)()
    bound = C.c_uint(0)
    assert L.b2rt_test_derived_arrays(ctx._h, sizes, None, None, None, None, None, C.byref(bound)) == 0
    arrs = [np.zeros(int(n), dtype=np.uint8) for n in sizes]
    assert L.b2rt_test_derived_arrays(ctx._h, sizes, *[a.ctypes.data for a in arrs], C.byref(bound)) == 0
    out = dict(zip(("wide", "leaf", "shade", "child_bin", "leaf_dir"), arrs))
    out["stack_bound"] = int(bound.value)
    out["scene_info"] = info
    return out


class DeviceTriangles:
    """Loader-order CLTriangles in a device buffer of `ctx` (b2rt_buffer_create + b2rt_device_pointer)."""

    def __init__(self, ctx, tris, capi):
        t = np.ascontiguousarray(tris)
        self.ctx, self.n = ctx, t.nbytes // 256
        buf, ptr, size = C.c_uint64(0), C.c_void_p(), C.c_size_t(0)
        ctx._ck(ctx._L.b2rt_buffer_create(ctx._h, capi.MEM_READ_ONLY | capi.MEM_COPY_HOST_PTR, t.nbytes, C.c_void_p(t.ctypes.data), C.byref(buf)))
        ctx._ck(ctx._L.b2rt_device_pointer(ctx._h, buf, C.byref(ptr), C.byref(size)))
        self.buf, self.ptr = buf.value, ptr.value

    def release(self):
        if self.buf:
            self.ctx._ck(self.ctx._L.b2rt_buffer_release(self.ctx._h, self.buf))
            self.buf = 0
