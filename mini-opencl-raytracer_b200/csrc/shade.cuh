// shade.cuh -- device re-statement of the per-pixel driver around the traversal:
// RNG, camera, BRDF sampling, lighting and accumulation of kernel_bvh.cl:57-96,
// 221-456. Not the optimisation target. Every fp32 operation replays the
// reference's operation order with one rounding per op; pow/sin/cos are evaluated
// in fp64 and rounded once, which reproduces glibc's (nearly always correctly
// rounded) powf/sinf/cosf used by the CPU oracle to within 1 ulp. Frames equal,
// bit for bit, the oracle built with these three functions in place of glibc's
// (tests/frame_oracle/oracle_devlibm.c, tests/test_gpu_frame_exact.py).
#pragma once
#include "traverse.cuh"

namespace b2rt {

struct V3 { float x, y, z; };
__device__ __forceinline__ V3 v3(float x, float y, float z) { V3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ V3 vadd(V3 a, V3 b) { return v3(xadd(a.x, b.x), xadd(a.y, b.y), xadd(a.z, b.z)); }
__device__ __forceinline__ V3 vsub(V3 a, V3 b) { return v3(xsub(a.x, b.x), xsub(a.y, b.y), xsub(a.z, b.z)); }
__device__ __forceinline__ V3 vmul(V3 a, V3 b) { return v3(xmul(a.x, b.x), xmul(a.y, b.y), xmul(a.z, b.z)); }
__device__ __forceinline__ V3 vscale(V3 a, float s) { return v3(xmul(a.x, s), xmul(a.y, s), xmul(a.z, s)); }
__device__ __forceinline__ V3 vdiv(V3 a, float s) { return v3(xdiv(a.x, s), xdiv(a.y, s), xdiv(a.z, s)); }
__device__ __forceinline__ V3 vneg(V3 a) { return v3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float vdot(V3 a, V3 b) { return xadd(xadd(xmul(a.x, b.x), xmul(a.y, b.y)), xmul(a.z, b.z)); }
__device__ __forceinline__ V3 vcross(V3 a, V3 b) {
    return v3(xsub(xmul(a.y, b.z), xmul(a.z, b.y)), xsub(xmul(a.z, b.x), xmul(a.x, b.z)), xsub(xmul(a.x, b.y), xmul(a.y, b.x)));
}
__device__ __forceinline__ V3 vnormalize(V3 a) { return vdiv(a, xsqrt(vdot(a, a))); }
__device__ __forceinline__ V3 ldv(const RefVec& p) { return v3(p.x, p.y, p.z); }

// powf as glibc evaluates it for the CPU oracle (correctly rounded except very near rounding boundaries): a double result
// good to ~1e-14 relative, rounded once to float. exp2(b * log2(a)) in fp64 delivers that at half the cost of CUDA's
// full double-precision pow(); the square (pow(x, 2.0), used twice by SampleBrdf) is exact in fp64 and also correct for
// negative x, where the logarithm route would give NaN. The logarithm route gives NaN where C99 powf returns 1 -- pow(x, 0)
// for x = 0, inf or NaN (0 * -inf, 0 * inf, 0 * NaN) and pow(1, y) for y = +-inf or NaN (inf * 0, NaN * 0) -- so those two
// cases return 1 first. SampleBrdf reaches both: roughness 0 gives the exponent 1/(alpha+1) = 0, roughness sqrt(2) gives
// alpha = -1 and the exponent inf, and rnd() returns exactly 0 or 1 for some seeds. For the bases the kernel passes
// (rnd() in [0, 1], pixel values >= 0 or NaN, any value squared) the other special values follow powf by themselves:
// pow(0, b>0) = 0, pow(0, b<0) = inf, pow(inf, b>0) = inf, pow(x<1, inf) = 0, NaN propagates. A negative base with an
// integer exponent other than 2 would not (NaN instead of +-|a|^b); no caller passes one.
__device__ __forceinline__ float pow_cr(float a, float b) {
    if (b == 0.0f || (a == 1.0f && !(fabsf(b) < INFINITY))) return 1.0f;   // folds away for a constant finite b
    if (b == 2.0f) return (float)((double)a * (double)a);
    return (float)exp2((double)b * log2((double)a));
}
__device__ __forceinline__ float sin_cr(float a) { return (float)sin((double)a); }
__device__ __forceinline__ float cos_cr(float a) { return (float)cos((double)a); }

// kernel_bvh.cl:57-71
__device__ __forceinline__ uint32_t hash_u32(uint32_t x) { return 1103515245u * x + 12345u; }
__device__ __forceinline__ float rnd(uint32_t& s) {
    s ^= s >> 16; s *= 0x7feb352dU; s ^= s >> 15; s *= 0x846ca68bU; s ^= s >> 16;
    return xdiv(__uint2float_rn(s), 4294967296.0f);   // (float)0xffffffffU rounds to 2^32
}

// CreateRay, kernel_bvh.cl:386-403 (returns the direction before InitRay normalises it again).
__device__ __forceinline__ V3 camera_dir(const FrameArgs& a, uint32_t gid, uint32_t& seed) {
    float inv_w = xdiv(1.0f, (float)a.width), inv_h = xdiv(1.0f, (float)a.height);
    float aspect = xdiv((float)a.width, (float)a.height);
    float x = xsub(xadd((float)(gid % a.width), rnd(seed)), 0.5f);
    float y = xsub(xadd((float)(gid / a.width), rnd(seed)), 0.5f);
    x = xmul(xmul(xsub(xmul(2.0f, xmul(xadd(x, 0.5f), inv_w)), 1.0f), a.angle), aspect);
    y = xmul(-xsub(1.0f, xmul(2.0f, xmul(xadd(y, 0.5f), inv_h))), a.angle);
    V3 front = v3(a.front[0], a.front[1], a.front[2]), up = v3(a.up[0], a.up[1], a.up[2]);
    return vnormalize(vadd(vadd(vscale(vcross(front, up), x), vscale(up, y)), front));
}

// kernel_bvh.cl:79-90 / 227-239 share this tail.
__device__ __forceinline__ V3 frame_sample(V3 n, float phi, float sin_theta, float cos_term) {
    V3 axis = fabsf(n.x) > 0.001f ? v3(0.0f, 1.0f, 0.0f) : v3(1.0f, 0.0f, 0.0f);
    V3 t = vnormalize(vcross(axis, n));
    V3 s = vcross(n, t);
    double sp, cp;
    sincos((double)phi, &sp, &cp);                       // sinf / cosf of the oracle: fp64 result rounded once (one range reduction for both)
    return vnormalize(vadd(vadd(vscale(vscale(s, (float)cp), sin_theta), vscale(vscale(t, (float)sp), sin_theta)),
                           vscale(n, cos_term)));
}

// SampleBrdf, kernel_bvh.cl:264-302 (GeometrySmith / FresnelSchlick results are unused by the reference).
__device__ __forceinline__ V3 sample_brdf(V3 wo, V3& wi, float& pdf, V3 normal, const RefMaterial& m, uint32_t& seed) {
    const float TWO_PI = 6.28318530718f, INV_PI = 0.31830988618f;
    if (rnd(seed) > 0.5f) {
        float alpha = xsub(xdiv(2.0f, pow_cr(m.roughness, 2.0f)), 2.0f);
        float phi = xmul(TWO_PI, rnd(seed));
        (void)rnd(seed);                                              // xi, drawn and unused (:230)
        float cos_theta = pow_cr(rnd(seed), xdiv(1.0f, xadd(alpha, 1.0f)));
        float sin_theta = xsqrt(max_cl(0.0f, xsub(1.0f, xmul(cos_theta, cos_theta))));
        V3 wh = frame_sample(normal, phi, sin_theta, cos_theta);
        wi = vadd(vneg(wo), vscale(wh, xmul(2.0f, vdot(wo, wh))));    // reflect(), :74-77
        if (xmul(vdot(wi, normal), vdot(wo, normal)) < 0.000001f) return v3(0.0f, 0.0f, 0.0f);
        float a2 = xmul(alpha, alpha);
        float D = xdiv(xmul(a2, INV_PI), pow_cr(xadd(xmul(xmul(cos_theta, cos_theta), xsub(a2, 1.0f)), 1.0f), 2.0f));
        pdf = xdiv(xmul(D, cos_theta), xmul(4.0f, max_cl(vdot(wo, wh), 0.0f)));
        float k = xdiv(D, xadd(xmul(xmul(4.0f, max_cl(vdot(wi, normal), 0.0f)), max_cl(vdot(wo, normal), 0.0f)), 0.001f));
        return v3(xmul(k, m.specular.x), xmul(k, m.specular.y), xmul(k, m.specular.z));
    }
    float phi = xmul(TWO_PI, rnd(seed));
    float sin2 = rnd(seed);
    wi = frame_sample(normal, phi, xsqrt(sin2), xsqrt(xsub(1.0f, sin2)));
    pdf = xmul(vdot(wi, normal), INV_PI);
    return vscale(ldv(m.diffuse), INV_PI);
}

// lightPixel, kernel_bvh.cl:304-347. (o,d,t) is the ray that produced the hit.
__device__ __forceinline__ float light_pixel(V3 o, V3 d, float t, V3 normal, int light_type) {
    V3 light_pos = v3(0.0f, -10.0f, 16.0f);
    float intensity = 1.0f, ndotl, attn = 1.0f;
    if (light_type <= 0) {
        ndotl = max_cl(vdot(normal, v3(0.5f, -0.4f, 0.1f)), 0.0f);
    } else {
        V3 X = vadd(o, vscale(d, t));
        V3 L = vsub(light_pos, X);
        ndotl = max_cl(vdot(normal, L), 0.0f);
        if (light_type == 1) {
            intensity = 16.0f;
            V3 eye = vsub(L, X);
            float dist = xsqrt(vdot(eye, eye));
            attn = (float)__ddiv_rn(1.0, (double)xmul(0.8f, xmul(dist, dist)));   // `1.0 /` is fp64 in the source (:335)
        }
    }
    return xmul(xmul(attn, intensity), ndotl);
}

// Interpolated shading normal of an accepted hit (kernel_bvh.cl:146).
__device__ __forceinline__ V3 hit_normal(const ShadeTri* shade, const HitX& h) {
    const U4* p = reinterpret_cast<const U4*>(shade + h.tri);
    U4 a = ld128(p), b = ld128(p + 1), c = ld128(p + 2);
    V3 n1 = v3(bits2f(a.x), bits2f(a.y), bits2f(a.z));
    V3 n2 = v3(bits2f(b.x), bits2f(b.y), bits2f(b.z));
    V3 n3 = v3(bits2f(c.x), bits2f(c.y), bits2f(c.z));
    float w = xsub(xsub(1.0f, h.u), h.v);
    return vnormalize(vadd(vadd(vscale(n2, h.u), vscale(n3, h.v)), vscale(n1, w)));
}

// Accumulation, kernel_bvh.cl:449-455.
// `mirror` (may be null): the same pixel of the root GPU's image in a multi-GPU frame. The running average is kept in the
// rank's own image (`px`, read and written locally); the finished value is stored through to the root as well, so the
// frame is complete there when the ranks' kernels end -- the gather is fused into the compute kernel's epilogue instead
// of a pack / all-gather / unpack sequence afterwards.
__device__ __forceinline__ void accumulate(float* px, float* mirror, V3 rad, uint32_t frame_count) {
    float4* out = reinterpret_cast<float4*>(px);
    if (frame_count == 0) {
        const float4 v0 = make_float4(pow_cr(rad.x, 0.45454545f), pow_cr(rad.y, 0.45454545f), pow_cr(rad.z, 0.45454545f), 0.0f);
        *out = v0;
        if (mirror) __stcs(reinterpret_cast<float4*>(mirror), v0);
        return;
    }
    float4 old = *out;
    float fm1 = __uint2float_rn(frame_count - 1u), fc = __uint2float_rn(frame_count);
    float r = pow_cr(xdiv(xadd(xmul(pow_cr(old.x, 2.2f), fm1), rad.x), fc), 0.454545f);
    float g = pow_cr(xdiv(xadd(xmul(pow_cr(old.y, 2.2f), fm1), rad.y), fc), 0.454545f);
    float b = pow_cr(xdiv(xadd(xmul(pow_cr(old.z, 2.2f), fm1), rad.z), fc), 0.454545f);
    *out = make_float4(r, g, b, 0.0f);
    if (mirror) __stcs(reinterpret_cast<float4*>(mirror), make_float4(r, g, b, 0.0f));
}

}  // namespace b2rt
