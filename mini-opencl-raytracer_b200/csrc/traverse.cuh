// traverse.cuh -- per-ray traversal primitives for the compressed wide BVH.
//
// Written once for the sm_100a kernels (kernels.cu). The same text also
// compiles as plain C++ (tests/emu/, TEST ONLY) so that the builder + traversal
// logic can be checked against the CPU oracle in a container with no GPU; the
// product library never contains or calls that host build.
//
// Exactness contract (SURVEY.md Appendix A):
//  * ray set-up, the leaf box gate and the Moller-Trumbore test replay the
//    reference's fp32 operation order with one IEEE rounding per operation
//    (no FMA contraction): InitRay kernel_bvh.cl:42-55, RayBounds :156-169,
//    RayTriangle :98-153. On the device every such op is an explicit
//    __f*_rn intrinsic, which nvcc never contracts, or a packed .rn.f32x2
//    op used under the rule at "packed fp32 pairs" below.
//  * leaves are entered in exactly the reference's DFS order (near child first
//    by sign[axis], kernel_bvh.cl:200-207) and a leaf's triangles are tested iff
//    the leaf's exact fp32 box passes RayBounds on [0, best]. Because a parent
//    box contains its children and fp32 subtraction/multiplication by a fixed
//    operand are monotone, that is equivalent to the reference's rule "every
//    ancestor passed when it was visited", so interior culling may be anything
//    conservative: here 8-bit quantised boxes evaluated with one FMA per plane and an
//    explicit error margin (see test_wide_node). For the same reason interior nodes may
//    be tested AHEAD of pending leaves with a stale (larger) `best` -- the Lane state
//    machine below keeps up to two leaves queued in order while it walks on.
#pragma once
#include "b2rt_types.h"

#ifndef B2_NODE_TEST_H2
#define B2_NODE_TEST_H2 1      // wide-node test in packed fp16 (two children per instruction); 0 = one fp32 FMA per plane
#endif
#ifndef B2_LEAF_QUEUE
#define B2_LEAF_QUEUE 2        // leaves a lane may hold back while it walks on (speculation depth)
#endif
#if defined(__CUDACC__)
#define B2_HD __device__ __forceinline__
#else
#define B2_HD inline
#include <cfenv>
#include <cmath>
#include <cstring>
#endif

namespace b2rt {

// ---- arithmetic primitives ----------------------------------------------------------
#if defined(__CUDACC__)
B2_HD float xadd(float a, float b) { return __fadd_rn(a, b); }
B2_HD float xsub(float a, float b) { return __fsub_rn(a, b); }
B2_HD float xmul(float a, float b) { return __fmul_rn(a, b); }
B2_HD float xdiv(float a, float b) { return __fdiv_rn(a, b); }
B2_HD float xsqrt(float a) { return __fsqrt_rn(a); }
B2_HD float sub_rd(float a, float b) { return __fsub_rd(a, b); }
B2_HD float sub_ru(float a, float b) { return __fsub_ru(a, b); }
B2_HD float fma_rd(float a, float b, float c) { return __fmaf_rd(a, b, c); }
B2_HD float fma_ru(float a, float b, float c) { return __fmaf_ru(a, b, c); }
B2_HD float mul_rd(float a, float b) { return __fmul_rd(a, b); }
B2_HD float mul_ru(float a, float b) { return __fmul_ru(a, b); }
B2_HD float max_nn(float a, float b) { return fmaxf(a, b); }   // NaN-ignoring
B2_HD float min_nn(float a, float b) { return fminf(a, b); }
B2_HD float u2f(uint32_t v) { return __uint2float_rn(v); }
B2_HD float fma_rn(float a, float b, float c) { return __fmaf_rn(a, b, c); }
// prmt.b32 without __byte_perm's selector masking; selectors used here never set a nibble's bit 3.
B2_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { uint32_t d; asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel)); return d; }

B2_HD uint32_t top_bit(uint32_t v) { return 31u - (uint32_t)__clz((int)v); }
B2_HD uint32_t low_mask(uint32_t n) { uint32_t d; asm("bmsk.clamp.b32 %0, %1, %2;" : "=r"(d) : "r"(0u), "r"(n)); return d; }   // (1 << n) - 1
B2_HD uint32_t byte_of(uint32_t w, uint32_t i) { return __byte_perm(w, 0, 0x4440u + i); }
B2_HD uint32_t popc32(uint32_t v) { return __popc(v); }
B2_HD uint32_t funnel_l(uint32_t lo, uint32_t hi, uint32_t n) { return __funnelshift_l(lo, hi, n); }
B2_HD float bits2f(uint32_t v) { return __uint_as_float(v); }
B2_HD uint32_t f2bits(float v) { return __float_as_uint(v); }
B2_HD U4 ld128(const U4* p) {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    U4 r; r.x = v.x; r.y = v.y; r.z = v.z; r.w = v.w; return r;
}
B2_HD uint32_t ld32(const uint32_t* p) { return __ldg(p); }
// warp collectives of the cooperative tail mode (coop.cuh); every lane of the warp calls them together
B2_HD uint32_t w_lane() { return threadIdx.x & 31u; }
B2_HD uint32_t w_ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
B2_HD uint32_t w_shfl(uint32_t v, uint32_t src) { return __shfl_sync(0xffffffffu, v, (int)src); }
B2_HD uint32_t w_redmin(uint32_t v) { return __reduce_min_sync(0xffffffffu, v); }
B2_HD uint32_t w_redor(uint32_t v) { return __reduce_or_sync(0xffffffffu, v); }
B2_HD void w_sync() { __syncwarp(); }
B2_HD uint32_t ctz32(uint32_t v) { return (uint32_t)__ffs((int)v) - 1u; }     // v != 0
B2_HD void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" :: "l"(p)); }
// packed fp16 arithmetic of test_wide_node_h2, on raw 32-bit patterns (two halves per register)
B2_HD uint32_t h2_fma(uint32_t a, uint32_t b, uint32_t c) { uint32_t d; asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); return d; }
B2_HD uint32_t h2_max(uint32_t a, uint32_t b) { uint32_t d; asm("max.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }   // NaN operand: the other one
B2_HD uint32_t h2_min(uint32_t a, uint32_t b) { uint32_t d; asm("min.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
B2_HD uint32_t h2_sub(uint32_t a, uint32_t b) { uint32_t d; asm("sub.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b)); return d; }
B2_HD uint32_t h2_both(float v) { uint32_t d; asm("cvt.rn.f16x2.f32 %0, %1, %1;" : "=r"(d) : "f"(v)); return d; }                   // (v, v) rounded to nearest; overflow -> inf
B2_HD uint32_t dot4(uint32_t a, uint32_t b) { return __dp4a(a, b, 0u); }                                                             // sum of byte products
__device__ unsigned long long g_stack_overflows;      // per device; read + cleared by b2rt_get_counters / b2rt_reset_counters
B2_HD void report_stack_overflow() { atomicAdd(&g_stack_overflows, 1ull); }
#else
// Host emulation (tests only). Built with -ffp-contract=off -frounding-math.
B2_HD float xadd(float a, float b) { volatile float r = a + b; return r; }
B2_HD float xsub(float a, float b) { volatile float r = a - b; return r; }
B2_HD float xmul(float a, float b) { volatile float r = a * b; return r; }
B2_HD float xdiv(float a, float b) { volatile float r = a / b; return r; }
B2_HD float xsqrt(float a) { return std::sqrt(a); }
template <class F> B2_HD float with_round(int mode, F f) {
    int old = std::fegetround(); std::fesetround(mode); volatile float r = f(); std::fesetround(old); return r;
}
B2_HD float sub_rd(float a, float b) { return with_round(FE_DOWNWARD, [&] { volatile float x = a, y = b; return x - y; }); }
B2_HD float sub_ru(float a, float b) { return with_round(FE_UPWARD, [&] { volatile float x = a, y = b; return x - y; }); }
B2_HD float fma_rd(float a, float b, float c) { return with_round(FE_DOWNWARD, [&] { volatile float x = a, y = b, z = c; return std::fmaf(x, y, z); }); }
B2_HD float fma_ru(float a, float b, float c) { return with_round(FE_UPWARD, [&] { volatile float x = a, y = b, z = c; return std::fmaf(x, y, z); }); }
B2_HD float mul_rd(float a, float b) { return with_round(FE_DOWNWARD, [&] { volatile float x = a, y = b; return x * y; }); }
B2_HD float mul_ru(float a, float b) { return with_round(FE_UPWARD, [&] { volatile float x = a, y = b; return x * y; }); }
B2_HD float max_nn(float a, float b) { return std::fmax(a, b); }
B2_HD float min_nn(float a, float b) { return std::fmin(a, b); }
B2_HD float u2f(uint32_t v) { return (float)v; }
B2_HD float fma_rn(float a, float b, float c) { return std::fmaf(a, b, c); }
B2_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {   // PTX prmt.b32, default mode: nibble bits 0-2 pick a byte, bit 3 replicates its sign
    uint64_t src = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t nib = (sel >> (4 * i)) & 0xfu;
        uint32_t byte = (uint32_t)((src >> (8 * (nib & 7u))) & 0xffu);
        if (nib & 8u) byte = (byte & 0x80u) ? 0xffu : 0u;
        r |= byte << (8 * i);
    }
    return r;
}
// IEEE binary16 on the host, enough for test_wide_node_h2: decode, round-to-nearest-even encode (subnormals, overflow to inf),
// and the packed operations with ONE rounding each (products and sums of halves are exact in double).
B2_HD double h_dec(uint32_t h) {
    const uint32_t s = (h >> 15) & 1u, e = (h >> 10) & 31u, m = h & 1023u;
    double v;
    if (e == 31u) v = m ? std::nan("") : INFINITY;
    else if (e == 0u) v = std::ldexp((double)m, -24);
    else v = std::ldexp((double)(m | 1024u), (int)e - 25);
    return s ? -v : v;
}
B2_HD uint32_t h_enc(double v) {
    if (std::isnan(v)) return 0x7fffu;
    const uint32_t s = std::signbit(v) ? 0x8000u : 0u;
    double a = std::fabs(v);
    if (a >= 65520.0) return s | 0x7c00u;                     // rounds to infinity
    if (a < std::ldexp(1.0, -14)) {                            // subnormal: multiples of 2^-24
        const double q = std::nearbyint(std::ldexp(a, 24));    // default rounding mode: to nearest even
        return s | (uint32_t)q;                                // 1024 -> the smallest normal, encoded correctly by the carry
    }
    int e;
    const double f = std::frexp(a, &e);                        // a = f * 2^e, f in [0.5, 1)
    double m = std::nearbyint(std::ldexp(f, 11));              // 11 significant bits
    if (m >= 2048.0) { m = 1024.0; ++e; }
    const int be = e - 1 + 15;
    if (be >= 31) return s | 0x7c00u;
    return s | ((uint32_t)be << 10) | ((uint32_t)m & 1023u);
}
template <class F> B2_HD uint32_t h2_map(uint32_t a, uint32_t b, uint32_t c, F f) {
    return h_enc(f(h_dec(a & 0xffffu), h_dec(b & 0xffffu), h_dec(c & 0xffffu))) | (h_enc(f(h_dec(a >> 16), h_dec(b >> 16), h_dec(c >> 16))) << 16);
}
B2_HD uint32_t h2_fma(uint32_t a, uint32_t b, uint32_t c) { return h2_map(a, b, c, [](double x, double y, double z) { return x * y + z; }); }
B2_HD uint32_t h2_sub(uint32_t a, uint32_t b) { return h2_map(a, b, 0u, [](double x, double y, double) { return x - y; }); }
B2_HD uint32_t h2_max(uint32_t a, uint32_t b) { return h2_map(a, b, 0u, [](double x, double y, double) { return std::fmax(x, y); }); }
B2_HD uint32_t h2_min(uint32_t a, uint32_t b) { return h2_map(a, b, 0u, [](double x, double y, double) { return std::fmin(x, y); }); }
B2_HD uint32_t h2_both(float v) { const uint32_t h = h_enc((double)v); return h | (h << 16); }
B2_HD uint32_t dot4(uint32_t a, uint32_t b) {
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r += ((a >> (8 * i)) & 0xffu) * ((b >> (8 * i)) & 0xffu);
    return r;
}
B2_HD uint32_t top_bit(uint32_t v) { return 31u - (uint32_t)__builtin_clz(v); }
B2_HD uint32_t low_mask(uint32_t n) { return n >= 32u ? 0xffffffffu : (1u << n) - 1u; }
B2_HD uint32_t byte_of(uint32_t w, uint32_t i) { return (w >> (8 * i)) & 0xffu; }
B2_HD uint32_t popc32(uint32_t v) { return (uint32_t)__builtin_popcount(v); }
B2_HD uint32_t funnel_l(uint32_t lo, uint32_t hi, uint32_t n) { return (uint32_t)(((((uint64_t)hi) << 32) | lo) << (n & 31u) >> 32); }
B2_HD float bits2f(uint32_t v) { float f; std::memcpy(&f, &v, 4); return f; }
B2_HD uint32_t f2bits(float v) { uint32_t u; std::memcpy(&u, &v, 4); return u; }
B2_HD U4 ld128(const U4* p) { return *p; }
B2_HD uint32_t ld32(const uint32_t* p) { return *p; }
}  // namespace b2rt
// Warp collectives on the host: tests/emu/warp_emu.cpp runs the 32 lanes of a warp as coroutines in lock step.
namespace b2rt_emu { uint32_t lane(); uint32_t exchange(uint32_t v, int op, uint32_t arg); }
namespace b2rt {
B2_HD uint32_t w_lane() { return b2rt_emu::lane(); }
B2_HD uint32_t w_ballot(bool p) { return b2rt_emu::exchange(p ? 1u : 0u, 0, 0); }
B2_HD uint32_t w_shfl(uint32_t v, uint32_t src) { return b2rt_emu::exchange(v, 1, src); }
B2_HD uint32_t w_redmin(uint32_t v) { return b2rt_emu::exchange(v, 2, 0); }
B2_HD uint32_t w_redor(uint32_t v) { return b2rt_emu::exchange(v, 3, 0); }
B2_HD void w_sync() { (void)b2rt_emu::exchange(0, 4, 0); }
B2_HD uint32_t ctz32(uint32_t v) { return (uint32_t)__builtin_ctz(v); }
B2_HD void prefetch_l2(const void*) {}
extern unsigned long long g_emu_stack_overflows;
extern unsigned long long g_emu_culling_violations;
B2_HD void report_stack_overflow() { ++g_emu_stack_overflows; }
#endif

// ---- packed fp32 pairs ----------------------------------------------------------------
// sm_100 evaluates add/sub/mul.rn.f32x2 as one FADD2 / FMUL2: two IEEE operations, each rounded on its own, in one issue
// slot. The exact leaf path (box_gate_exact, tri_eval_exact) runs on such pairs.
// HAZARD: ptxas contracts a mul.rn.f32x2 that feeds an add/sub.rn.f32x2 into one FFMA2 (one rounding instead of two) even
// under -fmad=false. So the halves of a packed product are only ever combined by scalar xadd / xsub (__fadd_rn /
// __fsub_rn, which are not contracted); packed sums may feed packed products. tests/test_packed_fp32_sass.py checks the SASS.
#if defined(__CUDACC__)
struct F2 { unsigned long long v; };      // one 64-bit register pair: half 0 in the low register
B2_HD F2 pack2(float a, float b) { F2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(a), "f"(b)); return r; }
B2_HD float lo2(F2 p) { float a; asm("mov.b64 {%0, _}, %1;" : "=f"(a) : "l"(p.v)); return a; }
B2_HD float hi2(F2 p) { float b; asm("mov.b64 {_, %0}, %1;" : "=f"(b) : "l"(p.v)); return b; }
B2_HD F2 sub2(F2 a, F2 b) { F2 r; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B2_HD F2 mul2(F2 a, F2 b) { F2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B2_HD F2 add2(F2 a, F2 b) { F2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v)); return r; }
B2_HD F2 fma2(F2 a, F2 b, F2 c) { F2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v)); return r; }   // two fma_rn
#else
// Host emulation: two scalar operations (the emulation cannot see a contraction; the SASS test does).
struct F2 { float a, b; };
B2_HD F2 pack2(float a, float b) { F2 r; r.a = a; r.b = b; return r; }
B2_HD float lo2(F2 p) { return p.a; }
B2_HD float hi2(F2 p) { return p.b; }
B2_HD F2 sub2(F2 x, F2 y) { return pack2(xsub(x.a, y.a), xsub(x.b, y.b)); }
B2_HD F2 mul2(F2 x, F2 y) { return pack2(xmul(x.a, y.a), xmul(x.b, y.b)); }
B2_HD F2 add2(F2 x, F2 y) { return pack2(xadd(x.a, y.a), xadd(x.b, y.b)); }
B2_HD F2 fma2(F2 x, F2 y, F2 z) { return pack2(fma_rn(x.a, y.a, z.a), fma_rn(x.b, y.b, z.b)); }
#endif
B2_HD F2 both2(float v) { return pack2(v, v); }
B2_HD F2 abs2(F2 p) { return pack2(fabsf(lo2(p)), fabsf(hi2(p))); }

// OpenCL max()/min() as worded by the spec ("y if x < y, otherwise x"), the
// convention the oracle pins for NaN operands (oracle/ref_build/cl_shim.hpp).
B2_HD float max_cl(float x, float y) { return x < y ? y : x; }
B2_HD float min_cl(float x, float y) { return y < x ? y : x; }

// ---- ray ----------------------------------------------------------------------------
struct RayX {
    float ox, oy, oz;
    float dx, dy, dz;      // normalised exactly like InitRay
    float ix, iy, iz;      // 1/d, may be +-inf
    uint32_t sign;         // bit a: inv[a] < 0; bit 3 (RAY_DEGENERATE): some inv[a] is infinite or beyond 2^100
};
enum : uint32_t { RAY_DEGENERATE = 8u };

// InitRay, kernel_bvh.cl:42-55, with normalize(v) = v / sqrt(dot(v,v)).
B2_HD RayX make_ray(float ox, float oy, float oz, float dx, float dy, float dz) {
    RayX r;
    float len = xsqrt(xadd(xadd(xmul(dx, dx), xmul(dy, dy)), xmul(dz, dz)));
    r.ox = ox; r.oy = oy; r.oz = oz;
    r.dx = xdiv(dx, len); r.dy = xdiv(dy, len); r.dz = xdiv(dz, len);
    r.ix = xdiv(1.0f, r.dx); r.iy = xdiv(1.0f, r.dy); r.iz = xdiv(1.0f, r.dz);
    r.sign = (r.ix < 0 ? 1u : 0u) | (r.iy < 0 ? 2u : 0u) | (r.iz < 0 ? 4u : 0u);
    // a direction component that is exactly (or all but) zero: 1/d is +-inf, the one-FMA plane evaluation of test_wide_node
    // then yields NaN on that axis (inf - inf) and stops culling there; such rays take test_wide_node_robust instead
    const float big = 1.2676506e30f;                       // 2^100
    if (!(fabsf(r.ix) <= big) || !(fabsf(r.iy) <= big) || !(fabsf(r.iz) <= big)) r.sign |= RAY_DEGENERATE;
    return r;
}

struct HitX {
    float t, u, v;
    uint32_t tri;          // B2RT_MISS (0xFFFFFFFF) until a triangle is accepted
};

struct TravCounters { uint32_t wide_nodes, leaf_blocks, leaf_pass, tri_tests, words, max_stack, rounds; };   // max_stack: most deferred references at once (incl. the register-held top)

// RayBounds, kernel_bvh.cl:156-169, on an exact fp32 box.
B2_HD bool box_gate_exact(const RayX& r, float lox, float loy, float loz, float hix, float hiy, float hiz, float best) {
    // (near, far) planes of an axis as one pair: a packed difference feeding a packed product is not contracted
    const F2 sx = mul2(sub2(pack2((r.sign & 1u) ? hix : lox, (r.sign & 1u) ? lox : hix), both2(r.ox)), both2(r.ix));
    const F2 sy = mul2(sub2(pack2((r.sign & 2u) ? hiy : loy, (r.sign & 2u) ? loy : hiy), both2(r.oy)), both2(r.iy));
    const F2 sz = mul2(sub2(pack2((r.sign & 4u) ? hiz : loz, (r.sign & 4u) ? loz : hiz), both2(r.oz)), both2(r.iz));
    float t0 = max_cl(0.0f, lo2(sx));
    float t1 = min_cl(best, hi2(sx));
    t0 = max_cl(t0, lo2(sy));
    t1 = min_cl(t1, hi2(sy));
    t0 = max_cl(t0, lo2(sz));
    t1 = min_cl(t1, hi2(sz));
    return t1 >= t0;
}

// RayTriangle, kernel_bvh.cl:98-153, for triangle (a,b,c) = (v1,v2,v3) with id `tri`.
// Accepts iff det >= 1e-8, 0<=u<=1, v>=0, u+v<=1 and t < best (no lower bound on t).
// Branch-free: the reference's early returns only skip work, so evaluating every comparison
// of the sequence and AND-ing them gives the same decision (NaN/inf operands included -- each
// comparison is the negation the reference tests, in its order) without divergent exits.
B2_HD bool tri_eval_exact(const RayX& r, float ax, float ay, float az, float bx, float by, float bz,
                          float cx, float cy, float cz, float& t, float& u, float& v) {
    // x and y of every vector form one pair (a vertex's x, y arrive adjacent from one 128-bit load), z stays scalar;
    // cross and dot products are FMUL2 whose halves are combined by scalar adds (see HAZARD)
    const F2 a = pack2(ax, ay), d = pack2(r.dx, r.dy);
    const F2 e1 = sub2(pack2(bx, by), a), e2 = sub2(pack2(cx, cy), a);
    const float e1z = xsub(bz, az), e2z = xsub(cz, az);
    const F2 m1 = mul2(d, both2(e2z)), m2 = mul2(e2, both2(r.dz)), m3 = mul2(d, pack2(hi2(e2), lo2(e2)));
    const F2 p = pack2(xsub(hi2(m1), hi2(m2)), xsub(lo2(m2), lo2(m1)));     // px = dy e2z - dz e2y, py = dz e2x - dx e2z
    const float pz = xsub(lo2(m3), hi2(m3));                                  // dx e2y - dy e2x
    const F2 m4 = mul2(e1, p);
    const float det = xadd(xadd(lo2(m4), hi2(m4)), xmul(e1z, pz));
    bool ok = !(det < 1.0e-8f) && !(-det > 1.0e-8f);                                   // :116
    const float inv = xdiv(1.0f, det);
    const F2 s = sub2(pack2(r.ox, r.oy), a);
    const float sz = xsub(r.oz, az);
    const F2 m5 = mul2(s, p);
    u = xmul(xadd(xadd(lo2(m5), hi2(m5)), xmul(sz, pz)), inv);
    ok = ok && !(u < 0.0f) && !(u > 1.0f);                                             // :125
    const F2 m6 = mul2(s, both2(e1z)), m7 = mul2(e1, both2(sz)), m8 = mul2(s, pack2(hi2(e1), lo2(e1)));
    const F2 q = pack2(xsub(hi2(m6), hi2(m7)), xsub(lo2(m7), lo2(m6)));     // qx = sy e1z - sz e1y, qy = sz e1x - sx e1z
    const float qz = xsub(lo2(m8), hi2(m8));                                  // sx e1y - sy e1x
    const F2 m9 = mul2(d, q);
    v = xmul(xadd(xadd(lo2(m9), hi2(m9)), xmul(r.dz, qz)), inv);
    ok = ok && !(v < 0.0f) && !(xadd(u, v) > 1.0f);                                    // :132
    const F2 m10 = mul2(e2, q);
    t = xmul(xadd(xadd(lo2(m10), hi2(m10)), xmul(e2z, qz)), inv);
    return ok;
}
B2_HD void tri_test_exact(const RayX& r, float ax, float ay, float az, float bx, float by, float bz,
                          float cx, float cy, float cz, uint32_t tri, HitX& h) {
    float t, u, v;
    const bool ok = tri_eval_exact(r, ax, ay, az, bx, by, bz, cx, cy, cz, t, u, v);
    if (ok && t < h.t) { h.t = t; h.u = u; h.v = v; h.tri = tri; }                      // :140
}

// ---- hit policies ------------------------------------------------------------------------
// HIT_CLOSEST: h is the nearest accepted hit. HIT_ANY: the walk ends at the first accepted hit.
// HIT_MULTI: the k nearest accepted hits, kept sorted by t in the ray's own output row (global memory, k records of 16 B);
// h then holds the list's state, so that the policy needs no register beyond the other two:
//     h.t   = bound: the ray's tmax while the row holds fewer than k hits, else the t of its k-th entry
//     h.u   = the ray's tmax (the value unused slots are padded with)
//     h.tri = the number of entries in the row
// A triangle is accepted iff RayTriangle accepts it with t < bound -- the closest-hit rule with `best` replaced by the
// bound, which never grows during the walk: the leaf gate on [0, bound] and every culling argument above carry over.
enum : int { HIT_CLOSEST = 0, HIT_ANY = 1, HIT_MULTI = 2 };
#if defined(__CUDACC__)
// The row is read back with an explicit coherent load: the same thread wrote it earlier in this launch, so the read-only
// path (ld.global.nc / __ldg) must not be used for it; the memory clobber keeps the load behind the stores before it.
B2_HD HitX ld_hit(const HitX* p) {
    HitX h; uint32_t t, u, v;
    asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(t), "=r"(u), "=r"(v), "=r"(h.tri) : "l"(p) : "memory");
    h.t = __uint_as_float(t); h.u = __uint_as_float(u); h.v = __uint_as_float(v);
    return h;
}
B2_HD void st_hit(HitX* p, float t, float u, float v, uint32_t tri) { *reinterpret_cast<float4*>(p) = make_float4(t, u, v, __uint_as_float(tri)); }
#else
B2_HD HitX ld_hit(const HitX* p) { return *p; }
B2_HD void st_hit(HitX* p, float t, float u, float v, uint32_t tri) { p->t = t; p->u = u; p->v = v; p->tri = tri; }
#endif
// Insert an accepted hit (t < h.t) into the row: after every entry with t' <= t, so equal t keeps visiting order like the
// reference's strict `<`; a full row drops its last entry. Entries only move here.
B2_HD void list_insert(HitX* row, uint32_t k, HitX& h, float t, float u, float v, uint32_t tri) {
    uint32_t j = h.tri < k ? h.tri : k - 1u;          // the slot that becomes occupied
    float last = t;                                    // what ends up in slot k - 1 (the new bound once the row is full)
    for (; j > 0u; --j) {
        const HitX p = ld_hit(row + j - 1u);
        if (!(p.t > t)) break;
        st_hit(row + j, p.t, p.u, p.v, p.tri);
        if (j == k - 1u) last = p.t;
    }
    st_hit(row + j, t, u, v, tri);
    if (h.tri < k) ++h.tri;
    if (h.tri == k) h.t = last;
}
B2_HD void tri_test_multi(const RayX& r, float ax, float ay, float az, float bx, float by, float bz,
                          float cx, float cy, float cz, uint32_t tri, HitX& h, HitX* row, uint32_t k) {
    float t, u, v;
    const bool ok = tri_eval_exact(r, ax, ay, az, bx, by, bz, cx, cy, cz, t, u, v);
    if (ok && t < h.t) list_insert(row, k, h, t, u, v, tri);
}
// A finished HIT_MULTI ray: slots [h.tri, k) of its row become {tmax, 0, 0, B2RT_MISS}.
B2_HD void pad_row(HitX* row, uint32_t k, const HitX& h) {
    for (uint32_t i = h.tri; i < k; ++i) st_hit(row + i, h.u, 0.0f, 0.0f, 0xFFFFFFFFu);
}

// ---- leaf block ----------------------------------------------------------------------
// The exact fp32 box of a one-record block: component-wise min / max of its vertices (exact operations; see b2rt_types.h).
B2_HD float min3_nn(float a, float b, float c) { return min_nn(min_nn(a, b), c); }
B2_HD float max3_nn(float a, float b, float c) { return max_nn(max_nn(a, b), c); }

// Returns true when at least one triangle was accepted by this call. MULTI: accepted hits go into `row` (HIT_MULTI).
template <bool COUNT, bool MULTI = false>
B2_HD bool visit_leaf(const U4* leaf, uint32_t offset, const RayX& r, HitX& h, TravCounters* c, HitX* row = nullptr, uint32_t row_len = 0) {
    const U4* p = leaf + offset;
    U4 a = ld128(p), b = ld128(p + 1), cc = ld128(p + 2);       // every block has >= 1 record
    const uint32_t nrec = (a.w >> LEAF_NREC_SHIFT) & LEAF_NREC_MASK;
    float lox, loy, loz, hix, hiy, hiz;
    if (a.w & LEAF_HAS_BOX) {                                   // rare: several records, or a box that is not the vertices' min / max
        const U4 b0 = ld128(p + LEAF_RECORD_WORDS * nrec), b1 = ld128(p + LEAF_RECORD_WORDS * nrec + 1);
        lox = bits2f(b0.x); loy = bits2f(b0.y); loz = bits2f(b0.z); hix = bits2f(b1.x); hiy = bits2f(b1.y); hiz = bits2f(b1.z);
        if (COUNT) c->words += LEAF_BOX_WORDS;
    } else {
        lox = min3_nn(bits2f(a.x), bits2f(b.x), bits2f(cc.x)); hix = max3_nn(bits2f(a.x), bits2f(b.x), bits2f(cc.x));
        loy = min3_nn(bits2f(a.y), bits2f(b.y), bits2f(cc.y)); hiy = max3_nn(bits2f(a.y), bits2f(b.y), bits2f(cc.y));
        loz = min3_nn(bits2f(a.z), bits2f(b.z), bits2f(cc.z)); hiz = max3_nn(bits2f(a.z), bits2f(b.z), bits2f(cc.z));
    }
    if (COUNT) { c->leaf_blocks++; c->words += LEAF_RECORD_WORDS * nrec; }
    if (!box_gate_exact(r, lox, loy, loz, hix, hiy, hiz, h.t))
        return false;
    if (COUNT) c->leaf_pass++;
    uint32_t before = h.tri;
    float t_before = h.t;
    uint32_t id = b.w;
    for (uint32_t k = 0;;) {
        float v1x = bits2f(a.x), v1y = bits2f(a.y), v1z = bits2f(a.z);
        float v2x = bits2f(b.x), v2y = bits2f(b.y), v2z = bits2f(b.z);
        float v3x = bits2f(cc.x), v3y = bits2f(cc.y), v3z = bits2f(cc.z);
        uint32_t flags = a.w & REC_FLAG_MASK;
        if (MULTI) tri_test_multi(r, v1x, v1y, v1z, v2x, v2y, v2z, v3x, v3y, v3z, id, h, row, row_len);
        else tri_test_exact(r, v1x, v1y, v1z, v2x, v2y, v2z, v3x, v3y, v3z, id, h);
        if (COUNT) c->tri_tests++;
        if (flags) {
            // the loader's second copy of the same triangle, rotated left (v2,v3,v1) or right (v3,v1,v2)
            const bool left = flags == REC_ROT_LEFT;
            if (MULTI) tri_test_multi(r, left ? v2x : v3x, left ? v2y : v3y, left ? v2z : v3z,
                                      left ? v3x : v1x, left ? v3y : v1y, left ? v3z : v1z,
                                      left ? v1x : v2x, left ? v1y : v2y, left ? v1z : v2z, id + 1, h, row, row_len);
            else tri_test_exact(r, left ? v2x : v3x, left ? v2y : v3y, left ? v2z : v3z,
                                left ? v3x : v1x, left ? v3y : v1y, left ? v3z : v1z,
                                left ? v1x : v2x, left ? v1y : v2y, left ? v1z : v2z, id + 1, h);
            if (COUNT) c->tri_tests++;
        }
        id += flags ? 2u : 1u;
        if (++k >= nrec) break;
        const U4* q = p + LEAF_RECORD_WORDS * k;
        a = ld128(q); b = ld128(q + 1); cc = ld128(q + 2);
    }
    return h.tri != before || h.t != t_before;
}

// ---- wide node ------------------------------------------------------------------------
struct WideHits {
    uint32_t mask;                // bit k: the child visited k-th (reference order) may intersect [0,best]
    uint32_t meta_lo, meta_hi;    // meta bytes permuted into visiting order
    uint32_t add_interior;        // child_base - META_INTERIOR
    uint32_t add_leaf;            // REF_LEAF_BIT | leaf_base
};

// Child reference of the child visited k-th: wide node index, or REF_LEAF_BIT | block offset.
// meta = 0x80 | index for interior children, block offset (< 0x80) for leaves, so ref = meta + addend.
B2_HD uint32_t child_ref(const WideHits& w, uint32_t k) {
    uint32_t m = prmt(w.meta_lo, w.meta_hi, k) & 0xffu;
    return m + ((m & META_INTERIOR) ? w.add_interior : w.add_leaf);
}

// float 1 + q * 2^-15 from byte i of w: the byte lands in mantissa bits 8..15 of 1.0f.
#define B2_PLANE_V(w, i) bits2f(prmt((w), one, 0x7604u | ((i) << 4)))

// Conservative slab test of the (up to) 8 quantised child boxes against [0, best], evaluated in
// the reference's visiting order for this ray's sign octant.
//
// With S = 2^(exp-127), plane(q) = base + q*S and v = 1 + q*2^-15, the reference's slab value for an
// exact plane P is R(P) = fl(fl(P - o) * inv) (kernel_bvh.cl:158-167). Here one FMA per plane gives
//     t(q) = fl(v*K + B),  K = 2^15*S*inv (exact), B = fl(A - K) -+ slack, A = fl(fl(base - o) * inv)
// whose real-arithmetic value is (plane(q) - o)*inv. Rounding of A, B and the FMA, plus the two
// roundings inside R, differ from that by less than 1.5 * 2^-22 * (|A| + |K|); slack =
// 2^-20 * (|A| + |K|) + 1e-35 therefore makes t_near(q_near) <= R(P) for every exact plane P on the
// far side of the quantised near plane (R is monotone in P), and likewise t_far >= R(P). NaNs
// (inv = +-inf or NaN, overflow) drop out of fminf/fmaxf, i.e. that axis does not constrain: the
// test can only pass more children than the reference's, never fewer.
B2_HD WideHits test_wide_node(const U4* wide, uint32_t index, const RayX& r, float best, uint32_t one) {
    const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * index;
    U4 w0 = ld128(p), w1 = ld128(p + 1), w2 = ld128(p + 2), w3 = ld128(p + 3), w4 = ld128(p + 4);
    const uint32_t order = ld32(reinterpret_cast<const uint32_t*>(p + 5) + r.sign);
    WideHits out;
    out.add_interior = w1.x - (uint32_t)META_INTERIOR;
    out.add_leaf = REF_LEAF_BIT | w1.y;
    const uint32_t sel_lo = order, sel_hi = order >> 16;      // prmt reads the low four nibbles only
    out.meta_lo = prmt(w1.z, w1.w, sel_lo);
    out.meta_hi = prmt(w1.z, w1.w, sel_hi);

    const float o[3] = { r.ox, r.oy, r.oz };
    const float inv[3] = { r.ix, r.iy, r.iz };
    const float base[3] = { bits2f(w0.x), bits2f(w0.y), bits2f(w0.z) };
    const uint32_t qlo_a[3] = { w2.x, w2.z, w3.x }, qlo_b[3] = { w2.y, w2.w, w3.y };   // slots 0..3 / 4..7
    const uint32_t qhi_a[3] = { w3.z, w4.x, w4.z }, qhi_b[3] = { w3.w, w4.y, w4.w };
    float K[3], Bn[3], Bf[3];
    uint32_t near_lo[3], near_hi[3], far_lo[3], far_hi[3];      // plane bytes in visiting order, ranks 0..3 / 4..7
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const uint32_t e = (w0.w >> (8 * a)) & 0xffu;
        K[a] = xmul(bits2f((e + 15u) << 23), inv[a]);
        const float A = xmul(xsub(base[a], o[a]), inv[a]);
        const float B = xsub(A, K[a]);
        const float slack = fma_rn(xadd(fabsf(A), fabsf(K[a])), 9.5367431640625e-7f, 1.0e-35f);
        Bn[a] = xsub(B, slack);
        Bf[a] = xadd(B, slack);
        const bool neg = (r.sign >> a) & 1u;
        const uint32_t na = neg ? qhi_a[a] : qlo_a[a], nb = neg ? qhi_b[a] : qlo_b[a];
        const uint32_t fa = neg ? qlo_a[a] : qhi_a[a], fb = neg ? qlo_b[a] : qhi_b[a];
        near_lo[a] = prmt(na, nb, sel_lo); near_hi[a] = prmt(na, nb, sel_hi);
        far_lo[a] = prmt(fa, fb, sel_lo);  far_hi[a] = prmt(fa, fb, sel_hi);
    }
    // Child k overlaps [0, best] iff F >= N, F >= 0 and best >= N with N = max(near planes), F = min(far planes)
    // (NaN planes drop out of fmaxf/fminf). All three are sign tests: the OR of the sign bits of F - N, F and
    // best - N says "cull", and one funnel shift per child collects it -- the two subtractions run on the FMA
    // pipe, which is idle next to the ALU pipe that PRMT/FMNMX keep busy. A NaN difference (inf - inf) has a
    // clear sign bit: the child is visited, which is always allowed (the exact leaf gate decides).
    uint32_t cull = 0;
#pragma unroll
    for (int kk = 7; kk >= 0; --kk) {
        const uint32_t k = (uint32_t)kk, i = k & 3u;
        float n0 = fma_rn(B2_PLANE_V(k < 4 ? near_lo[0] : near_hi[0], i), K[0], Bn[0]);
        float n1 = fma_rn(B2_PLANE_V(k < 4 ? near_lo[1] : near_hi[1], i), K[1], Bn[1]);
        float n2 = fma_rn(B2_PLANE_V(k < 4 ? near_lo[2] : near_hi[2], i), K[2], Bn[2]);
        float f0 = fma_rn(B2_PLANE_V(k < 4 ? far_lo[0] : far_hi[0], i), K[0], Bf[0]);
        float f1 = fma_rn(B2_PLANE_V(k < 4 ? far_lo[1] : far_hi[1], i), K[1], Bf[1]);
        float f2 = fma_rn(B2_PLANE_V(k < 4 ? far_lo[2] : far_hi[2], i), K[2], Bf[2]);
        const float N = max_nn(max_nn(n0, n1), n2);
        const float F = min_nn(min_nn(f0, f1), f2);
        const uint32_t bad = f2bits(xsub(F, N)) | f2bits(F) | f2bits(xsub(best, N));
        cull = funnel_l(bad, cull, 1);                      // cull = cull << 1 | sign(bad): child 0 ends up in bit 0
    }
    const uint32_t mask = ~cull & 0xffu;
    out.mask = mask & ((1u << (w0.w >> 24)) - 1u);
    return out;
}

B2_HD WideHits test_wide_node_robust(const U4* wide, uint32_t index, const RayX& r, float best);

// Packed-fp16 variant of test_wide_node (B2_NODE_TEST_H2): two children per instruction.
//
// The slab values are evaluated RELATIVE to t_ref (the ray's entry distance into the node's own box, any fp32 number would
// do) and SCALED by a power of two chosen per visit, so that they fit binary16: with K1 = S*inv (exact), A = fl(fl(base-o)*inv)
//     T(q) = ((A - t_ref) + q*K1) * scale            plane q of this axis, real arithmetic
// and scale = 2^(117 - exponent(max_a |K1|)), the largest |K2| = |K1| * 2^24 * scale lies in [2^14, 2^15) and the node's own
// extent in T is below 255 * 2^-9.5 < 1. One PRMT turns two plane bytes into two SUBNORMAL halves q * 2^-24 (byte in the
// low mantissa bits, exponent zero: exact), one fma.f16x2 gives q*2^-24 * K2h + Bh for both children.
// Error budget per plane, against the reference's R(P) = fl(fl(P - o) * inv) of any exact plane beyond the quantised one:
//   K2h = K2 (1 + d), |d| <= 2^-11:  q*2^-24*|K2|*2^-11 <= 2^-16 |K2| * 2^-11 * 255/256 ... < 2^-11 * 2^-16 |K2| * 256
//   Bh rounded to nearest: 2^-11 |B|;   the FMA's own rounding: 2^-11 (|B| + 2^-16 |K2|) (or 2^-25 absolute when subnormal);
//   fp32 roundings inside A, A - t_ref and R(P): < 2^-21 (|A| + |t_ref|) * scale.
// Their sum is below 2^-10 (|Bh| + 2^-16 |K2|) + 2^-21 (...) with |Bh| <= |B| + slack, so
// slack = 1.025 * 2^-10 (|B| + 2^-16 |K2|) + 2^-20 (max_a |A| + |t_ref|) scale + 2^-22 covers it; near planes are lowered and far
// planes raised by it before the conversion. Overflowing values become +-inf on the side that keeps the test
// conservative: a near plane beyond the binary16 range is more than 2^5 node extents past the entry point while some far
// plane of the node is within 255 * max|K1| of it, so the child is truly missed; a far plane below the range lies before the
// entry point, likewise; inf - inf = NaN has a clear sign bit and lets the child through.
// 0 and `best` join the same frame (rounded outwards): pass iff min(far..., best) >= max(near..., 0).
// Children are evaluated in SLOT order; the 8 sign bytes are permuted into visiting order afterwards (two PRMT) and
// squeezed into the mask with two dot products.
B2_HD WideHits test_wide_node_h2(const U4* wide, uint32_t index, const RayX& r, float best) {
    const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * index;
    U4 w0 = ld128(p), w1 = ld128(p + 1), w2 = ld128(p + 2), w3 = ld128(p + 3), w4 = ld128(p + 4);
    const uint32_t order = ld32(reinterpret_cast<const uint32_t*>(p + 5) + r.sign);
    WideHits out;
    out.add_interior = w1.x - (uint32_t)META_INTERIOR;
    out.add_leaf = REF_LEAF_BIT | w1.y;
    const uint32_t sel_lo = order, sel_hi = order >> 16;
    out.meta_lo = prmt(w1.z, w1.w, sel_lo);
    out.meta_hi = prmt(w1.z, w1.w, sel_hi);

    const uint32_t qlo_a[3] = { w2.x, w2.z, w3.x }, qlo_b[3] = { w2.y, w2.w, w3.y };   // slots 0..3 / 4..7
    const uint32_t qhi_a[3] = { w3.z, w4.x, w4.z }, qhi_b[3] = { w3.w, w4.y, w4.w };
    // From B on, the fp32 set-up runs with x and y as one packed pair (xy) and z scalar: the same operations with the same
    // roundings, except where ptxas contracts a packed product into the packed sum it feeds (see "packed fp32 pairs"). The
    // only such products here are by scale, a power of two: exact unless the result is subnormal or overflows. A
    // contraction therefore drops a rounding that was nothing or below 2^-149; the error budget above already counts that
    // rounding as one of its terms, so the slack still covers the contracted sequence. An overflowing B gives slack = inf
    // and Bn / Bf = -inf / +inf instead of NaN / +inf: the near plane still drops out of the max and the far one out of the
    // min. The fallback guard reads the scalar A and K1, which are not contracted.
    // K1 and A stay scalar: packing the ray's origin and reciprocal into pairs costs more moves and registers (spills in
    // trace_persistent) than the two paired products save
    const float o[3] = { r.ox, r.oy, r.oz };
    const float inv[3] = { r.ix, r.iy, r.iz };
    const float base[3] = { bits2f(w0.x), bits2f(w0.y), bits2f(w0.z) };
    float K1[3], A[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        K1[a] = xmul(bits2f(((w0.w >> (8 * a)) & 0xffu) << 23), inv[a]);
        A[a] = xmul(xsub(base[a], o[a]), inv[a]);
    }
    const F2 K1xy = pack2(K1[0], K1[1]), Axy = pack2(A[0], A[1]);
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
    const float e32 = fma_rn(xmul(xadd(amax, t_ref), scale), 9.5367431640625e-7f, 2.384185791015625e-7f);   // the fp32 roundings' share, one bound for all axes
    const F2 Bxy = mul2(sub2(Axy, both2(t_ref)), both2(scale));
    const F2 K2xy = mul2(K1xy, both2(kscale));
    const F2 Sxy = fma2(fma2(abs2(K2xy), both2(1.52587890625e-5f), abs2(Bxy)), both2(1.0009765625e-3f), both2(e32));
    const F2 Bnxy = sub2(Bxy, Sxy), Bfxy = add2(Bxy, Sxy);
    const float Bz = xmul(xsub(A[2], t_ref), scale), K2z = xmul(K1[2], kscale);
    const float Sz = fma_rn(fma_rn(fabsf(K2z), 1.52587890625e-5f, fabsf(Bz)), 1.0009765625e-3f, e32);
    const uint32_t Kh[3] = { h2_both(lo2(K2xy)), h2_both(hi2(K2xy)), h2_both(K2z) };
    const uint32_t Bn[3] = { h2_both(lo2(Bnxy)), h2_both(hi2(Bnxy)), h2_both(xsub(Bz, Sz)) };
    const uint32_t Bf[3] = { h2_both(lo2(Bfxy)), h2_both(hi2(Bfxy)), h2_both(xadd(Bz, Sz)) };
    // 0 and best as one pair (-z, b), z = -t_ref * scale, b = (best - t_ref) * scale: both moved up by 2^-10 of their
    // magnitude + 2^-22, i.e. z lowered and b raised, one conversion each
    const F2 zb = mul2(pack2(t_ref, xsub(best, t_ref)), both2(scale));
    const F2 zbs = add2(zb, fma2(abs2(zb), both2(9.765625e-4f), both2(2.384185791015625e-7f)));
    const uint32_t zero_h = h2_both(-lo2(zbs)), best_h = h2_both(hi2(zbs));
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

// The same decision for rays whose reciprocal direction has an infinite (or NaN, or > 2^100) component (RAY_DEGENERATE):
// a direction component of exactly zero is not rare in rendered frames (a few rays per million: central camera rows,
// BRDF frames of axis-aligned normals), and with one FMA per plane such an axis evaluates to inf - inf = NaN and no longer
// culls -- the ray then walks every node its projection onto the other axes overlaps (measured: 26 000 steps instead of
// ~40, a 5 ms tail on a 4 ms frame share). Here the planes are decoded to fp32 (rounded outwards: lo_q <= base + q*S <=
// child's exact lo as real numbers, wide_bvh.cpp) and the reference's own two operations fl(fl(P - o) * inv) are applied:
// they are monotone in P, so near(lo_q) <= near(exact box of any leaf below) and far(hi_q) >= far(...); (P - o) * inf is
// +-inf on the correct side and 0 * inf = NaN drops out of fmaxf/fminf like out of the reference's max()/min().
B2_HD WideHits test_wide_node_robust(const U4* wide, uint32_t index, const RayX& r, float best) {
    const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * index;
    U4 w0 = ld128(p), w1 = ld128(p + 1), w2 = ld128(p + 2), w3 = ld128(p + 3), w4 = ld128(p + 4);
    const uint32_t order = ld32(reinterpret_cast<const uint32_t*>(p + 5) + (r.sign & 7u));
    WideHits out;
    out.add_interior = w1.x - (uint32_t)META_INTERIOR;
    out.add_leaf = REF_LEAF_BIT | w1.y;
    out.meta_lo = prmt(w1.z, w1.w, order);
    out.meta_hi = prmt(w1.z, w1.w, order >> 16);
    const float o[3] = { r.ox, r.oy, r.oz };
    const float inv[3] = { r.ix, r.iy, r.iz };
    const float base[3] = { bits2f(w0.x), bits2f(w0.y), bits2f(w0.z) };
    const uint32_t qlo_a[3] = { w2.x, w2.z, w3.x }, qlo_b[3] = { w2.y, w2.w, w3.y };
    const uint32_t qhi_a[3] = { w3.z, w4.x, w4.z }, qhi_b[3] = { w3.w, w4.y, w4.w };
    uint32_t mask = 0;
    const uint32_t n_children = w0.w >> 24;
    for (uint32_t k = 0; k < n_children; ++k) {
        const uint32_t slot = (order >> (4u * k)) & 7u;
        float N = 0.0f, F = best;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float S = bits2f(((w0.w >> (8 * a)) & 0xffu) << 23);
            const float lo = fma_rd(u2f(prmt(qlo_a[a], qlo_b[a], slot) & 0xffu), S, base[a]);
            const float hi = fma_ru(u2f(prmt(qhi_a[a], qhi_b[a], slot) & 0xffu), S, base[a]);
            const bool neg = (r.sign >> a) & 1u;
            N = max_nn(N, xmul(xsub(neg ? hi : lo, o[a]), inv[a]));
            F = min_nn(F, xmul(xsub(neg ? lo : hi, o[a]), inv[a]));
        }
        if (F >= N) mask |= 1u << k;
    }
    out.mask = mask;
    return out;
}

// ---- the short stack -------------------------------------------------------------------------
// Lane<> reaches its stack of deferred child references only through stk_get / stk_set, so that the caller chooses where
// the entries live: a plain local array (the per-ray driver below, the frame megakernel, the host emulation), or
// HybridStack -- the first B2_SMEM_STACK entries in shared memory, one 4-byte column per thread (conflict-free), the rest in
// the local array at the same indices. Measured on the bench stream (host emulation, depth histogram at pop time): 26 % of
// the pops find the stack empty, 69 % read one of the first six entries, 4.5 % a deeper one -- while ncu saw 38 % of the
// local-memory pops miss L1 (the lines are evicted by the node / leaf traffic between a push and its pop) and local memory
// make up a quarter of the kernel's L2 sectors. Six entries x 128 threads x 8 CTAs = 24 KB per SM, inside the 32 KB
// shared-memory carve-out the kernel already ran with: L1 keeps its size.
B2_HD uint32_t stk_get(const uint32_t* s, int i) { return s[i]; }
B2_HD void stk_set(uint32_t* s, int i, uint32_t v) { s[i] = v; }
template <int DEPTH, int STRIDE>
struct HybridStack {
    uint32_t* sh;          // this thread's column: entry i at sh[i * STRIDE]
    uint32_t* loc;         // entries DEPTH.. (indices as in a plain array)
};
template <int DEPTH, int STRIDE> B2_HD uint32_t stk_get(HybridStack<DEPTH, STRIDE> s, int i) { return i < DEPTH ? s.sh[i * STRIDE] : s.loc[i]; }
template <int DEPTH, int STRIDE> B2_HD void stk_set(HybridStack<DEPTH, STRIDE> s, int i, uint32_t v) { if (i < DEPTH) s.sh[i * STRIDE] = v; else s.loc[i] = v; }

// ---- one ray's traversal state ------------------------------------------------------------
// node_step() tests the current wide node and walks on; leaves met on the way are queued (two
// slots, FIFO) and consumed in order by leaf_step(). Any interleaving of the two calls that the
// wants_*() predicates allow gives the reference's result; the kernels pick per warp, by vote,
// whichever step more lanes are waiting for.
// The short stack of child references lives OUTSIDE this struct (a plain local array owned by the
// caller): with the array inside, the compiler keeps every scalar of the struct in local memory too.
// P: hit policy (HIT_CLOSEST, HIT_ANY, HIT_MULTI).
template <int P, bool COUNT, int CAP>
struct Lane {
    static constexpr bool ANY = P == HIT_ANY, MULTI = P == HIT_MULTI;
    RayX r;
    HitX h;
    uint32_t cur;          // wide node to test next, a leaf waiting for a queue slot, or REF_EMPTY
    uint32_t leaf0, leaf1; // queued leaves, leaf0 first
#if B2_LEAF_QUEUE == 3
    uint32_t leaf2;
#endif
    uint32_t top;          // most recently pushed child reference, kept in a register (REF_EMPTY = stack empty)
    int sp;                // entries below `top`, in the caller's local array
    bool overflow;
    TravCounters tc;

    B2_HD void start(const RayX& ray, float tmax) {
        r = ray;
        h.t = tmax; h.u = 0.0f; h.v = 0.0f; h.tri = 0xFFFFFFFFu;
        if (MULTI) { h.u = tmax; h.tri = 0u; }        // empty list (see HIT_MULTI)
        cur = 0; leaf0 = leaf1 = top = REF_EMPTY; sp = 0; overflow = false;
#if B2_LEAF_QUEUE == 3
        leaf2 = REF_EMPTY;
#endif
    }
    B2_HD void clear() {
        cur = leaf0 = leaf1 = top = REF_EMPTY; sp = 0;
#if B2_LEAF_QUEUE == 3
        leaf2 = REF_EMPTY;
#endif
    }
    B2_HD bool done() const { return cur == REF_EMPTY && leaf0 == REF_EMPTY; }
    B2_HD bool wants_node() const { return cur != REF_EMPTY && !(cur & REF_LEAF_BIT); }
    B2_HD bool wants_leaf() const { return leaf0 != REF_EMPTY; }

    // The top of the stack sits in a register: a pop answers at once and the load that refills the
    // register from local memory is only waited for by the NEXT pop.
    template <class S> B2_HD void push(S stack, uint32_t ref) {
        // CAP is at least the tree's exact bound (wide_stack_bound, checked at upload), so the else branch never runs. The
        // flag is only READ by the counting build (-> b2rt_counters::stack_overflows): in the production build it is dead
        // and costs nothing -- an atomic or a live flag here measurably slows the loop (r2 A/B: -4 %).
        if (COUNT) { if (top != REF_EMPTY) { if (sp < CAP) stk_set(stack, sp++, top); else overflow = true; } }
        else {
            // branch-free: the slot at sp is free by construction (sp < CAP, see above), so the old top is stored
            // unconditionally and only kept (sp advanced) when there was one
            stk_set(stack, sp, top);
            sp += top != REF_EMPTY ? 1 : 0;
        }
        top = ref;
        if (COUNT && (uint32_t)sp + 1u > tc.max_stack) tc.max_stack = (uint32_t)sp + 1u;
    }
    template <class S> B2_HD uint32_t pop(S stack) {
        uint32_t ref = top;
        if (sp > 0) { --sp; top = stk_get(stack, sp); } else top = REF_EMPTY;
        return ref;
    }
    // Move leaves from `cur` into the queue while there is room.
    template <class S> B2_HD void settle(S stack) {
#if B2_LEAF_QUEUE == 3
        while (cur != REF_EMPTY && (cur & REF_LEAF_BIT) && leaf2 == REF_EMPTY) {
            if (leaf0 == REF_EMPTY) leaf0 = cur; else if (leaf1 == REF_EMPTY) leaf1 = cur; else leaf2 = cur;
            cur = pop(stack);
        }
#else
        while (cur != REF_EMPTY && (cur & REF_LEAF_BIT) && leaf1 == REF_EMPTY) {
            if (leaf0 == REF_EMPTY) leaf0 = cur; else leaf1 = cur;
            cur = pop(stack);
        }
#endif
    }
    // A suspended ray comes back (two-step tail, kernels.cu): F[0..n) is its frontier as coop_dump laid it out (front =
    // F[n-1]); the entries are dealt out again the way settle() would have left them -- queued leaves, current node,
    // register-held top, the rest on the short stack (never more entries there than the first owner had). The caller has
    // called start() and restored h.
    B2_HD void resume(uint32_t* stack, const uint32_t* F, uint32_t n) {
        leaf0 = leaf1 = REF_EMPTY;
        cur = n ? F[--n] : REF_EMPTY;
        while (cur != REF_EMPTY && (cur & REF_LEAF_BIT) && leaf1 == REF_EMPTY) {
            if (leaf0 == REF_EMPTY) leaf0 = cur; else leaf1 = cur;
            cur = n ? F[--n] : REF_EMPTY;
        }
        top = n ? F[--n] : REF_EMPTY;
        sp = (int)n;
        for (uint32_t i = 0; i < n; ++i) stack[i] = F[i];
    }
    // `one` must be 0x3F800000, passed as run-time data: held in one register it lets the constant
    // byte selectors of B2_PLANE_V be instruction immediates (ptxas otherwise keeps four selector registers).
    template <class S> B2_HD void node_step(const U4* wide, S stack, uint32_t one) {
#if B2_NODE_TEST_H2
        WideHits w = (r.sign & RAY_DEGENERATE) ? test_wide_node_robust(wide, cur, r, h.t) : test_wide_node_h2(wide, cur, r, h.t);
#else
        WideHits w = (r.sign & RAY_DEGENERATE) ? test_wide_node_robust(wide, cur, r, h.t) : test_wide_node(wide, cur, r, h.t, one);
#endif
#if defined(B2_EMU_CHECK_CULLING)
        // host emulation only: no child that the exact-arithmetic test lets through may be culled by the fast one
        { const WideHits x = test_wide_node_robust(wide, cur, r, h.t); if (x.mask & ~w.mask) ++g_emu_culling_violations; }
#endif
        if (COUNT) { tc.wide_nodes++; tc.words += WIDE_NODE_WORDS; }
        uint32_t m = w.mask;
        if (m == 0) { cur = pop(stack); }
        else {
            while (m & (m - 1u)) {                       // more than one: push the farthest
                uint32_t k = top_bit(m);
                m &= low_mask(k);
                push(stack, child_ref(w, k));
            }
            cur = child_ref(w, top_bit(m));
        }
        settle(stack);
    }
    // Returns true when the ray is finished by this leaf (any-hit accept, or best < 0: every later
    // box test of the reference fails, SURVEY.md Appendix A-5; for HIT_MULTI the bound < 0).
    // row, k: the ray's output row and its length (HIT_MULTI only).
    template <class S> B2_HD bool leaf_step(const U4* leaf, S stack, HitX* row = nullptr, uint32_t k = 0) {
        bool got = visit_leaf<COUNT, MULTI>(leaf, leaf0 & ~REF_LEAF_BIT, r, h, COUNT ? &tc : nullptr, row, k);
#if B2_LEAF_QUEUE == 3
        leaf0 = leaf1; leaf1 = leaf2; leaf2 = REF_EMPTY;
#else
        leaf0 = leaf1; leaf1 = REF_EMPTY;
#endif
        if ((ANY && got) || h.t < 0.0f) { clear(); return true; }
        settle(stack);
        return false;
    }
};

// ---- simple per-ray driver (one thread = one ray; also the host emulation) -------------
// `schedule` != 0 makes the emulation pick node/leaf steps pseudo-randomly whenever both are
// allowed, to exercise every interleaving the warp-vote kernels can produce.
// HIT_MULTI: the hits go to row[0, k), padded when the ray is finished.
template <int P, bool COUNT, int CAP>
B2_HD HitX trace_wide(const U4* wide, const U4* leaf, const RayX& r, float tmax, TravCounters* c, bool* overflow,
                      uint32_t one, uint32_t schedule = 0, HitX* row = nullptr, uint32_t k = 0) {
    Lane<P, COUNT, CAP> L;
    uint32_t stack[CAP];
    L.tc.wide_nodes = L.tc.leaf_blocks = L.tc.leaf_pass = L.tc.tri_tests = L.tc.words = L.tc.max_stack = L.tc.rounds = 0;
    L.start(r, tmax);
    while (!L.done()) {
        const bool node = L.wants_node(), lf = L.wants_leaf();
        bool do_leaf = lf;                                  // default: consume pending leaves first (no speculation)
        if (node && lf && schedule) { schedule = schedule * 1664525u + 1013904223u; do_leaf = (schedule >> 16) & 1u; }
        if (do_leaf) { if (L.leaf_step(leaf, stack, row, k)) break; }
        else L.node_step(wide, stack, one);
    }
    if (P == HIT_MULTI) pad_row(row, k, L.h);
    if (COUNT && c) *c = L.tc;
    if (overflow) *overflow = L.overflow;
    return L.h;
}

}  // namespace b2rt
