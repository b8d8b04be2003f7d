"""The packed-fp32 set-up of the wide-node test (test_wide_node_h2) must stay within its written slack argument and pay off.

traverse.cuh evaluates the node test's per-axis fp32 set-up with x and y as one packed pair. Culling only has to stay
conservative, and the comment above the set-up argues that a contraction of a packed product into the packed sum it feeds
(ptxas does this even under -fmad=false) is covered by the slack: the only packed products that feed packed sums are the
products by `scale`, a power of two. This test compiles the node test with the library's own nvcc flags and reads the SASS:
- at most one FFMA2 per explicit packed fma (three) plus one per packed sum fed by a product by `scale` (three);
- fewer instructions than the same test with the all-scalar set-up it replaced (kept below as the reference).
Needs nvcc and cuobjdump, not a GPU."""
import os
import shutil
import subprocess

import pytest

from test_packed_fp32_sass import _nvcc_flags, _opcodes

PROBE = r"""
#include "traverse.cuh"
using namespace b2rt;

// the all-scalar set-up (one fp32 operation per axis and step)
__device__ __forceinline__ WideHits node_scalar(const U4* wide, uint32_t index, const RayX& r, float best) {
    const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * index;
    U4 w0 = ld128(p), w1 = ld128(p + 1), w2 = ld128(p + 2), w3 = ld128(p + 3), w4 = ld128(p + 4);
    const uint32_t order = ld32(reinterpret_cast<const uint32_t*>(p + 5) + r.sign);
    WideHits out;
    out.add_interior = w1.x - (uint32_t)META_INTERIOR;
    out.add_leaf = REF_LEAF_BIT | w1.y;
    const uint32_t sel_lo = order, sel_hi = order >> 16;
    out.meta_lo = prmt(w1.z, w1.w, sel_lo);
    out.meta_hi = prmt(w1.z, w1.w, sel_hi);

    const float o[3] = { r.ox, r.oy, r.oz };
    const float inv[3] = { r.ix, r.iy, r.iz };
    const float base[3] = { bits2f(w0.x), bits2f(w0.y), bits2f(w0.z) };
    const uint32_t qlo_a[3] = { w2.x, w2.z, w3.x }, qlo_b[3] = { w2.y, w2.w, w3.y };   // slots 0..3 / 4..7
    const uint32_t qhi_a[3] = { w3.z, w4.x, w4.z }, qhi_b[3] = { w3.w, w4.y, w4.w };
    float K1[3], A[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        K1[a] = xmul(bits2f(((w0.w >> (8 * a)) & 0xffu) << 23), inv[a]);
        A[a] = xmul(xsub(base[a], o[a]), inv[a]);
    }
    const float kmax = max_nn(max_nn(fabsf(K1[0]), fabsf(K1[1])), fabsf(K1[2]));
    // magnitudes this frame cannot hold (overflow of (base - o) * inv or S * inv: coordinates or reciprocals beyond 2^100):
    // decide in fp32 instead. Written so that NaN takes the branch too.
    const float amax = max_nn(max_nn(fabsf(A[0]), fabsf(A[1])), fabsf(A[2]));
    if (!(max_nn(amax, xmul(kmax, 256.0f)) < 1.2676506e30f))
        return test_wide_node_robust(wide, index, r, best);
    // entry distance into the node's box (near plane = q 0 or q 255 by the ray's sign), clamped at 0
    const float t_ref = max_nn(max_nn(max_nn((r.sign & 1u) ? fma_rn(255.0f, K1[0], A[0]) : A[0], (r.sign & 2u) ? fma_rn(255.0f, K1[1], A[1]) : A[1]),
                                      (r.sign & 4u) ? fma_rn(255.0f, K1[2], A[2]) : A[2]), 0.0f);
    uint32_t eb = f2bits(kmax) >> 23;                                   // biased exponent (kmax >= 0, finite: degenerate rays never get here)
    eb = eb < 15u ? 15u : eb;                                           // |K1| below 2^-112: keep the scale factors representable
    const float scale = bits2f((244u - eb) << 23);                     // 2^(117 - (eb - 127))
    const float kscale = bits2f((268u - eb) << 23);                    // scale * 2^24
    uint32_t Kh[3], Bn[3], Bf[3];
    const float e32 = fma_rn(xmul(xadd(amax, t_ref), scale), 9.5367431640625e-7f, 2.384185791015625e-7f);   // the fp32 roundings' share, one bound for all axes
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float B = xmul(xsub(A[a], t_ref), scale);
        const float K2 = xmul(K1[a], kscale);
        const float slack = fma_rn(fma_rn(fabsf(K2), 1.52587890625e-5f, fabsf(B)), 1.0009765625e-3f, e32);
        Kh[a] = h2_both(K2);
        Bn[a] = h2_both(xsub(B, slack));
        Bf[a] = h2_both(xadd(B, slack));
    }
    const float z = xmul(-t_ref, scale), b = xmul(xsub(best, t_ref), scale);
    const uint32_t zero_h = h2_both(xsub(z, fma_rn(fabsf(z), 9.765625e-4f, 2.384185791015625e-7f)));     // 0 and best: one conversion each, 2^-11 relative
    const uint32_t best_h = h2_both(xadd(b, fma_rn(fabsf(b), 9.765625e-4f, 2.384185791015625e-7f)));
    uint32_t d[4];
#pragma unroll
    for (int pr = 0; pr < 4; ++pr) {
        // slots 2pr, 2pr+1: bytes (0,1) or (2,3) of the word that holds them, each widened to a subnormal half
        const uint32_t sel = (pr & 1) ? 0x4342u : 0x4140u;
        uint32_t N = zero_h, F = best_h;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const bool neg = (r.sign >> a) & 1u;
            const uint32_t lo_w = pr < 2 ? qlo_a[a] : qlo_b[a], hi_w = pr < 2 ? qhi_a[a] : qhi_b[a];
            const uint32_t qn = prmt(neg ? hi_w : lo_w, 0u, sel), qf = prmt(neg ? lo_w : hi_w, 0u, sel);
            N = h2_max(N, h2_fma(qn, Kh[a], Bn[a]));
            F = h2_min(F, h2_fma(qf, Kh[a], Bf[a]));
        }
        d[pr] = h2_sub(F, N);                                           // sign bit set: the child is culled
    }
    // sign bytes of the eight differences in slot order (0xff = culled), then in visiting order, then one bit each
    const uint32_t c_lo = prmt(d[0], d[1], 0xfdb9u), c_hi = prmt(d[2], d[3], 0xfdb9u);
    const uint32_t v_lo = prmt(c_lo, c_hi, sel_lo), v_hi = prmt(c_lo, c_hi, sel_hi);
    const uint32_t cull = dot4(v_lo & 0x08040201u, 0x01010101u) | (dot4(v_hi & 0x08040201u, 0x01010101u) << 4);
    out.mask = ~cull & ((1u << (w0.w >> 24)) - 1u);
    return out;
}

extern "C" __global__ void probe_packed(const U4* wide, const RayX* rays, const float* best, uint32_t* out) {
    const uint32_t i = threadIdx.x;
    const WideHits w = test_wide_node_h2(wide, 7u * i, rays[i], best[i]);
    out[3 * i] = w.mask; out[3 * i + 1] = w.meta_lo; out[3 * i + 2] = w.meta_hi;
}
extern "C" __global__ void probe_scalar(const U4* wide, const RayX* rays, const float* best, uint32_t* out) {
    const uint32_t i = threadIdx.x;
    const WideHits w = node_scalar(wide, 7u * i, rays[i], best[i]);
    out[3 * i] = w.mask; out[3 * i + 1] = w.meta_lo; out[3 * i + 2] = w.meta_hi;
}
"""

EXPLICIT_FMA2 = 3          # the two slack terms of the xy pair, the margin of the (0, best) pair
CONTRACTIBLE_SUMS = 3      # Bn and Bf of the xy pair, the (0, best) pair plus its margin


def test_node_setup_packed_within_slack_argument(tmp_path):
    nvcc, flags = _nvcc_flags()
    if not (os.path.exists(nvcc) or shutil.which(nvcc)) or shutil.which("cuobjdump") is None:
        pytest.skip("needs nvcc and cuobjdump")
    src = tmp_path / "node_probe.cu"
    src.write_text(PROBE)
    cubin = tmp_path / "node_probe.cubin"
    subprocess.run([nvcc] + flags + ["-cubin", "-o", str(cubin), str(src)], check=True, capture_output=True, text=True)
    sass = subprocess.run(["cuobjdump", "-sass", str(cubin)], check=True, capture_output=True, text=True).stdout
    packed, scalar = _opcodes(sass, "probe_packed"), _opcodes(sass, "probe_scalar")
    assert packed["FMUL2"] > 0 and packed["FADD2"] > 0, "the node test no longer runs packed fp32: %s" % dict(packed)
    assert scalar["FFMA2"] == 0 and scalar["FMUL2"] == 0 and scalar["FADD2"] == 0
    assert packed["FFMA2"] <= EXPLICIT_FMA2 + CONTRACTIBLE_SUMS, "more FFMA2 than the slack argument covers: %s" % dict(packed)
    n_packed, n_scalar = sum(packed.values()), sum(scalar.values())
    assert n_packed < n_scalar, "the packed set-up is not shorter (%d >= %d instructions)" % (n_packed, n_scalar)
