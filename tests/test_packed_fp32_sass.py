"""The exact leaf path's packed fp32 arithmetic (FADD2 / FMUL2) must keep one rounding per operation.

ptxas contracts a mul.rn.f32x2 that feeds an add/sub.rn.f32x2 into one FFMA2 even under -fmad=false, and the host
emulation (which runs a packed operation as two scalar ones) cannot see that. So this test compiles the box gate and the
Moller-Trumbore test of traverse.cuh with the library's own nvcc flags and reads the SASS: no FFMA2 at all, and no more
scalar FFMA than the same sequence written with scalar intrinsics (the __fdiv_rn expansion has FFMAs of its own).
Needs nvcc and cuobjdump, not a GPU."""
import collections
import importlib.util
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT

PKG = os.path.join(ROOT, "mini-opencl-raytracer_b200")

PROBE = r"""
#include "traverse.cuh"
using namespace b2rt;

// the reference's scalar sequence (RayBounds + RayTriangle), one __f*_rn per operation
__device__ __forceinline__ bool gate_scalar(const RayX& r, const float* b, float best) {
    float nx = (r.sign & 1u) ? b[3] : b[0], fx = (r.sign & 1u) ? b[0] : b[3];
    float ny = (r.sign & 2u) ? b[4] : b[1], fy = (r.sign & 2u) ? b[1] : b[4];
    float nz = (r.sign & 4u) ? b[5] : b[2], fz = (r.sign & 4u) ? b[2] : b[5];
    float t0 = max_cl(0.0f, xmul(xsub(nx, r.ox), r.ix)), t1 = min_cl(best, xmul(xsub(fx, r.ox), r.ix));
    t0 = max_cl(t0, xmul(xsub(ny, r.oy), r.iy)); t1 = min_cl(t1, xmul(xsub(fy, r.oy), r.iy));
    t0 = max_cl(t0, xmul(xsub(nz, r.oz), r.iz)); t1 = min_cl(t1, xmul(xsub(fz, r.oz), r.iz));
    return t1 >= t0;
}
__device__ __forceinline__ bool tri_scalar(const RayX& r, const float* v, float& t, float& u, float& w) {
    float e1x = xsub(v[3], v[0]), e1y = xsub(v[4], v[1]), e1z = xsub(v[5], v[2]);
    float e2x = xsub(v[6], v[0]), e2y = xsub(v[7], v[1]), e2z = xsub(v[8], v[2]);
    float px = xsub(xmul(r.dy, e2z), xmul(r.dz, e2y)), py = xsub(xmul(r.dz, e2x), xmul(r.dx, e2z));
    float pz = xsub(xmul(r.dx, e2y), xmul(r.dy, e2x));
    float det = xadd(xadd(xmul(e1x, px), xmul(e1y, py)), xmul(e1z, pz));
    float inv = xdiv(1.0f, det);
    float tx = xsub(r.ox, v[0]), ty = xsub(r.oy, v[1]), tz = xsub(r.oz, v[2]);
    u = xmul(xadd(xadd(xmul(tx, px), xmul(ty, py)), xmul(tz, pz)), inv);
    float qx = xsub(xmul(ty, e1z), xmul(tz, e1y)), qy = xsub(xmul(tz, e1x), xmul(tx, e1z));
    float qz = xsub(xmul(tx, e1y), xmul(ty, e1x));
    w = xmul(xadd(xadd(xmul(r.dx, qx), xmul(r.dy, qy)), xmul(r.dz, qz)), inv);
    t = xmul(xadd(xadd(xmul(e2x, qx), xmul(e2y, qy)), xmul(e2z, qz)), inv);
    return !(det < 1.0e-8f) && !(-det > 1.0e-8f) && !(u < 0.0f) && !(u > 1.0f) && !(w < 0.0f) && !(xadd(u, w) > 1.0f);
}
__device__ __forceinline__ RayX probe_ray(const float* in) {
    RayX r;
    r.ox = in[0]; r.oy = in[1]; r.oz = in[2]; r.dx = in[3]; r.dy = in[4]; r.dz = in[5];
    r.ix = in[6]; r.iy = in[7]; r.iz = in[8]; r.sign = __float_as_uint(in[9]);
    return r;
}
extern "C" __global__ void probe_packed(const float* in, float* out) {
    const float* p = in + 16 * threadIdx.x;
    const RayX r = probe_ray(p);
    float t, u, v;
    const bool g = box_gate_exact(r, p[10], p[11], p[12], p[13], p[14], p[15], p[16]);
    const bool ok = tri_eval_exact(r, p[17], p[18], p[19], p[20], p[21], p[22], p[23], p[24], p[25], t, u, v);
    out[4 * threadIdx.x] = t; out[4 * threadIdx.x + 1] = u; out[4 * threadIdx.x + 2] = v;
    out[4 * threadIdx.x + 3] = (g ? 1.0f : 0.0f) + (ok ? 2.0f : 0.0f);
}
extern "C" __global__ void probe_scalar(const float* in, float* out) {
    const float* p = in + 16 * threadIdx.x;
    const RayX r = probe_ray(p);
    float t, u, v;
    const bool g = gate_scalar(r, p + 10, p[16]);
    const bool ok = tri_scalar(r, p + 17, t, u, v);
    out[4 * threadIdx.x] = t; out[4 * threadIdx.x + 1] = u; out[4 * threadIdx.x + 2] = v;
    out[4 * threadIdx.x + 3] = (g ? 1.0f : 0.0f) + (ok ? 2.0f : 0.0f);
}
"""


def _nvcc_flags():
    spec = importlib.util.spec_from_file_location("_b2rt_build_flags", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.NVCC, [f for f in mod.NVCC_FLAGS if f != "-Xcompiler" and not f.startswith("-fPIC")]


def _opcodes(sass, kernel):
    body = re.split(r"\n\s*Function : ", sass)
    text = next(b for b in body if b.split("\n", 1)[0].strip() == kernel)
    ops = collections.Counter()
    for line in text.splitlines():
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_]+)", line)
        if m:
            ops[m.group(1)] += 1
    return ops


def test_exact_leaf_path_has_no_contracted_packed_products(tmp_path):
    nvcc, flags = _nvcc_flags()
    if not (os.path.exists(nvcc) or shutil.which(nvcc)) or shutil.which("cuobjdump") is None:
        pytest.skip("needs nvcc and cuobjdump")
    src = tmp_path / "probe.cu"
    src.write_text(PROBE)
    cubin = tmp_path / "probe.cubin"
    subprocess.run([nvcc] + flags + ["-cubin", "-o", str(cubin), str(src)], check=True, capture_output=True, text=True)
    sass = subprocess.run(["cuobjdump", "-sass", str(cubin)], check=True, capture_output=True, text=True).stdout
    packed, scalar = _opcodes(sass, "probe_packed"), _opcodes(sass, "probe_scalar")
    assert packed["FMUL2"] > 0 and packed["FADD2"] > 0, "the probe no longer exercises packed fp32: %s" % dict(packed)
    assert packed["FFMA2"] == 0, "a packed product was contracted into FFMA2"
    assert packed["FFMA"] <= scalar["FFMA"], "more FFMA than the scalar sequence (%d > %d): a product was contracted" % (
        packed["FFMA"], scalar["FFMA"])
    assert scalar["FFMA2"] == 0 and scalar["FMUL2"] == 0
