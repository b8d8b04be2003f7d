// shade_probe.cu -- TEST INFRASTRUCTURE ONLY: the frame kernels' shading functions (csrc/shade.cuh, compiled with the
// product's nvcc flags) run one record per thread on the device, so that each can be compared bit for bit with the
// oracle's function of the same name (tests/frame_oracle/oracle_devlibm.c, fo_run). A record is 16 input words and
// 16 output words; the layouts below are those of fo_record.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstring>

#include "shade.cuh"

namespace {
using namespace b2rt;

enum { OP_POW = 0, OP_SINCOS = 1, OP_FRAME = 2, OP_BRDF = 3, OP_LIGHT = 4, OP_CAMERA = 5, OP_RND = 6, OP_ACCUMULATE = 7 };

__device__ float wf(const uint32_t* w, int k) { return __uint_as_float(w[k]); }
__device__ V3 ldw(const uint32_t* w) { return v3(wf(w, 0), wf(w, 1), wf(w, 2)); }
__device__ void stw(uint32_t* w, V3 v) { w[0] = __float_as_uint(v.x); w[1] = __float_as_uint(v.y); w[2] = __float_as_uint(v.z); }

__global__ void probe_kernel(int op, uint64_t n, const uint32_t* __restrict__ all_in, uint32_t* __restrict__ all_out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* in = all_in + 16 * i;
    uint32_t* out = all_out + 16 * i;
    for (int k = 0; k < 16; ++k) out[k] = 0u;
    switch (op) {
    case OP_POW:                      // a, b -> pow_cr(a, b)
        out[0] = __float_as_uint(pow_cr(wf(in, 0), wf(in, 1)));
        break;
    case OP_SINCOS:                   // a -> sin_cr(a), cos_cr(a)
        out[0] = __float_as_uint(sin_cr(wf(in, 0)));
        out[1] = __float_as_uint(cos_cr(wf(in, 0)));
        break;
    case OP_FRAME:                    // n[3], phi, sin_theta, cos_term -> frame_sample
        stw(out, frame_sample(ldw(in), wf(in, 3), wf(in, 4), wf(in, 5)));
        break;
    case OP_BRDF: {                   // wo[3], normal[3], roughness, specular[3], diffuse[3], seed -> f[3], wi[3], pdf, seed
        RefMaterial m;
        memset(&m, 0, sizeof(m));
        m.roughness = wf(in, 6);
        m.specular.x = wf(in, 7); m.specular.y = wf(in, 8); m.specular.z = wf(in, 9);
        m.diffuse.x = wf(in, 10); m.diffuse.y = wf(in, 11); m.diffuse.z = wf(in, 12);
        uint32_t seed = in[13];
        V3 wi = v3(0.0f, 0.0f, 0.0f);
        float pdf = 0.0f;
        stw(out, sample_brdf(ldw(in), wi, pdf, ldw(in + 3), m, seed));
        stw(out + 3, wi);
        out[6] = __float_as_uint(pdf); out[7] = seed;
        break;
    }
    case OP_LIGHT:                    // o[3], d[3], t, normal[3], light_type -> light_pixel
        out[0] = __float_as_uint(light_pixel(ldw(in), ldw(in + 3), wf(in, 6), ldw(in + 7), (int)in[10]));
        break;
    case OP_CAMERA: {                 // width, height, gid, seed, angle, front[3], up[3] -> InitRay's direction, seed
        FrameArgs a;
        memset(&a, 0, sizeof(a));
        a.width = in[0]; a.height = in[1]; a.angle = wf(in, 4);
        for (int k = 0; k < 3; ++k) { a.front[k] = wf(in, 5 + k); a.up[k] = wf(in, 8 + k); }
        uint32_t seed = in[3];
        const V3 d = camera_dir(a, in[2], seed);
        const RayX r = make_ray(0.0f, 0.0f, 0.0f, d.x, d.y, d.z);
        stw(out, v3(r.dx, r.dy, r.dz));
        out[3] = seed;
        break;
    }
    case OP_RND: {                    // seed -> rnd(seed), the advanced seed, hash_u32(seed)
        uint32_t seed = in[0];
        out[0] = __float_as_uint(rnd(seed));
        out[1] = seed;
        out[2] = hash_u32(in[0]);
        break;
    }
    case OP_ACCUMULATE: {             // old pixel[4], radiance[3], frame_count -> new pixel[4]
        float4 px = make_float4(wf(in, 0), wf(in, 1), wf(in, 2), wf(in, 3));
        accumulate(&px.x, nullptr, ldw(in + 4), in[7]);
        out[0] = __float_as_uint(px.x); out[1] = __float_as_uint(px.y); out[2] = __float_as_uint(px.z); out[3] = __float_as_uint(px.w);
        break;
    }
    default:
        break;
    }
}
}  // namespace

// n records of 16 words at host addresses `in` / `out`. Returns a cudaError_t.
extern "C" int shade_probe_run(int op, uint64_t n, const uint32_t* in, uint32_t* out) {
    if (n == 0) return 0;
    const size_t bytes = 16 * sizeof(uint32_t) * n;
    uint32_t *d_in = nullptr, *d_out = nullptr;
    cudaError_t e = cudaMalloc(&d_in, bytes);
    if (e == cudaSuccess) e = cudaMalloc(&d_out, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(d_in, in, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        probe_kernel<<<(unsigned)((n + 127) / 128), 128>>>(op, n, d_in, d_out);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d_in);
    cudaFree(d_out);
    return (int)e;
}
