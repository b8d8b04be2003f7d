// refit.cu -- b2rt_refit_scene: new vertex data for the bound scene, same topology. Everything the kernels read is
// refreshed ON THE DEVICE, no tree is rebuilt (SURVEY.md 8f-2 "build / refit"; the reference can only re-run
// CLBVHScene::RecursiveBuild, CLBVHnode.cpp:7-159, and upload again):
//   1. the new CLTriangle array replaces the bound triangle buffer (one H2D copy);
//   2. refit_leaf_kernel   binary leaves: box of their triangles (the same min/max chain as CLBVHnode.cpp:190-193);
//                          parent links of the pre-order node array;
//   3. refit_up_kernel     interior boxes bottom-up (second arrival at a node unions its children), written into the bound
//                          CLLinearBVHNode buffer -- b2rt_read_buffer returns the refitted tree in the reference's format;
//   4. refit_wide_kernel   every wide node re-quantises its child boxes (new frame origin / exponents / 8-bit planes,
//                          conservative like wide_bvh.cpp); treelet shape, child references and visiting orders stay;
//   5. refit_block_kernel  leaf blocks: exact leaf box and vertex positions; a record that stood for the loader's two
//                          copies of a triangle must still do so (else the call fails: rebuild instead);
//   6. refit_shade_kernel  per-triangle normals and material index.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>
#include <string>
#include "context.h"

using namespace b2rt;
using namespace b2rt_detail;

namespace {

enum : unsigned { REFIT_ERR_NONFINITE = 1u, REFIT_ERR_DUPLICATE = 2u, REFIT_ERR_RANGE = 4u, REFIT_ERR_LEAF_BOX = 8u };

__global__ void refit_leaf_kernel(RefNode* __restrict__ nodes, uint32_t n_nodes, const RefTriangle* __restrict__ tris, int* __restrict__ parent,
                                  unsigned* __restrict__ arrivals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    arrivals[i] = 0u;
    if (i == 0) parent[0] = -1;
    RefNode& nd = nodes[i];
    if (nd.nPrimitives == 0) { parent[i + 1] = (int)i; parent[nd.offset] = (int)i; return; }
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (uint32_t t = nd.offset; t < nd.offset + nd.nPrimitives; ++t) {
        const RefVec* p[3] = { &tris[t].v1.position, &tris[t].v2.position, &tris[t].v3.position };
        for (int k = 0; k < 3; ++k) {
            lo[0] = fminf(lo[0], p[k]->x); lo[1] = fminf(lo[1], p[k]->y); lo[2] = fminf(lo[2], p[k]->z);
            hi[0] = fmaxf(hi[0], p[k]->x); hi[1] = fmaxf(hi[1], p[k]->y); hi[2] = fmaxf(hi[2], p[k]->z);
        }
    }
    nd.bmin.x = lo[0]; nd.bmin.y = lo[1]; nd.bmin.z = lo[2];
    nd.bmax.x = hi[0]; nd.bmax.y = hi[1]; nd.bmax.z = hi[2];
}

__global__ void refit_up_kernel(RefNode* __restrict__ nodes, uint32_t n_nodes, const int* __restrict__ parent, unsigned* __restrict__ arrivals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes || nodes[i].nPrimitives == 0) return;
    int node = parent[i];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&arrivals[node], 1u) == 0u) return;              // the second arrival sees both children done
        const float* a = reinterpret_cast<const float*>(&nodes[node + 1]);
        const float* b = reinterpret_cast<const float*>(&nodes[nodes[node].offset]);
        float* d = reinterpret_cast<float*>(&nodes[node]);
        // children were written by other threads of this launch: read them past L1
        for (int k = 0; k < 3; ++k) {
            d[k] = fminf(__ldcg(a + k), __ldcg(b + k));
            d[4 + k] = fmaxf(__ldcg(a + 4 + k), __ldcg(b + 4 + k));
        }
        node = parent[node];
    }
}

// Largest q in [0,255] with base + q*s <= lo, resp. smallest q with base + q*s >= hi (as real numbers); the float
// operands are exact in double, their difference is unless the exponents are far apart -- then one step is given away.
__device__ int quant_floor_d(float base, double s, float lo) {
    double q = floor(((double)lo - (double)base) / s);
    if (lo != 0.0f && base != 0.0f && abs(ilogbf(lo) - ilogbf(base)) > 24) q -= 1.0;
    return (int)fmin(fmax(q, 0.0), 255.0);
}
__device__ int quant_ceil_d(float base, double s, float hi) {
    double q = ceil(((double)hi - (double)base) / s);
    if (hi != 0.0f && base != 0.0f && abs(ilogbf(hi) - ilogbf(base)) > 24) q += 1.0;
    return (int)fmin(fmax(q, 0.0), 1000.0);                             // > 255 tells the caller to widen the grid
}

__global__ void refit_wide_kernel(WideNode* __restrict__ wide, uint32_t n_wide, const uint32_t* __restrict__ child_bin, const RefNode* __restrict__ nodes,
                                  unsigned* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_wide) return;
    WideNode wn = wide[i];
    const int n = wn.n_children;
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    float cl[8][3], ch[8][3];
    for (int c = 0; c < n; ++c) {
        const RefNode& b = nodes[child_bin[8 * (size_t)i + c]];
        cl[c][0] = b.bmin.x; cl[c][1] = b.bmin.y; cl[c][2] = b.bmin.z; ch[c][0] = b.bmax.x; ch[c][1] = b.bmax.y; ch[c][2] = b.bmax.z;
        for (int a = 0; a < 3; ++a) { lo[a] = fminf(lo[a], cl[c][a]); hi[a] = fmaxf(hi[a], ch[c][a]); }
    }
    for (int a = 0; a < 3; ++a) {
        if (!(lo[a] <= hi[a]) || !isfinite(lo[a]) || !isfinite(hi[a])) { atomicOr(error, REFIT_ERR_NONFINITE); return; }
        wn.base[a] = lo[a];
        int e = 1;
        const double extent = (double)hi[a] - (double)lo[a];
        if (extent > 0.0) { int k; (void)frexp(extent / 255.0, &k); e = min(max(k + 127, 1), 254); }
        for (;; ++e) {
            if (e > 230) { atomicOr(error, REFIT_ERR_RANGE); return; }
            const double s = ldexp(1.0, e - 127);
            bool ok = true;
            for (int c = 0; c < 8 && ok; ++c) {
                if (c >= n) { wn.qlo[a][c] = 255; wn.qhi[a][c] = 0; continue; }
                const int ql = quant_floor_d(lo[a], s, cl[c][a]), qh = quant_ceil_d(lo[a], s, ch[c][a]);
                if (qh > 255) { ok = false; break; }
                wn.qlo[a][c] = (uint8_t)ql;
                wn.qhi[a][c] = (uint8_t)qh;
            }
            if (ok) { wn.exp[a] = (uint8_t)e; break; }
        }
    }
    wide[i] = wn;
}

__device__ __forceinline__ bool same_bits(const RefVec& a, const RefVec& b) {
    return __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y) && __float_as_uint(a.z) == __float_as_uint(b.z);
}

__global__ void refit_block_kernel(U4* __restrict__ leaf, const uint32_t* __restrict__ leaf_dir, uint32_t n_blocks, const RefNode* __restrict__ nodes,
                                   const RefTriangle* __restrict__ tris, unsigned* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_blocks) return;
    const RefNode& nd = nodes[leaf_dir[2 * (size_t)i]];
    U4* p = leaf + leaf_dir[2 * (size_t)i + 1];
    const uint32_t head = p[0].w, nrec = (head >> LEAF_NREC_SHIFT) & LEAF_NREC_MASK;
    uint32_t id = p[1].w;
    const uint32_t first = id;
    for (uint32_t k = 0; k < nrec; ++k) {
        U4* q = p + LEAF_RECORD_WORDS * k;
        const uint32_t w0 = q[0].w, flags = w0 & REC_FLAG_MASK;
        const RefTriangle& t = tris[id];
        if (flags) {
            // the record stands for triangle id AND its rotated copy id + 1: the new data must keep them bit-identical
            const RefTriangle& s = tris[id + 1];
            const bool ok = flags == REC_ROT_LEFT ? (same_bits(s.v1.position, t.v2.position) && same_bits(s.v2.position, t.v3.position) && same_bits(s.v3.position, t.v1.position))
                                                  : (same_bits(s.v1.position, t.v3.position) && same_bits(s.v2.position, t.v1.position) && same_bits(s.v3.position, t.v2.position));
            if (!ok) atomicOr(error, REFIT_ERR_DUPLICATE);
        }
        q[0] = U4{ __float_as_uint(t.v1.position.x), __float_as_uint(t.v1.position.y), __float_as_uint(t.v1.position.z), w0 };
        q[1] = U4{ __float_as_uint(t.v2.position.x), __float_as_uint(t.v2.position.y), __float_as_uint(t.v2.position.z), k == 0 ? first : 0u };
        q[2] = U4{ __float_as_uint(t.v3.position.x), __float_as_uint(t.v3.position.y), __float_as_uint(t.v3.position.z), 0u };
        id += flags ? 2u : 1u;
    }
    // A block without a stored box relies on box == min / max of its vertices; refit_leaf_kernel has just recomputed the
    // node's box as exactly that (a NaN vertex would break the equality: reported, the scene must be uploaded afresh).
    if (head & LEAF_HAS_BOX) {
        U4* q = p + LEAF_RECORD_WORDS * nrec;
        q[0] = U4{ __float_as_uint(nd.bmin.x), __float_as_uint(nd.bmin.y), __float_as_uint(nd.bmin.z), 0u };
        q[1] = U4{ __float_as_uint(nd.bmax.x), __float_as_uint(nd.bmax.y), __float_as_uint(nd.bmax.z), 0u };
    } else {
        const RefTriangle& t = tris[first];
        const float lo[3] = { fminf(fminf(t.v1.position.x, t.v2.position.x), t.v3.position.x), fminf(fminf(t.v1.position.y, t.v2.position.y), t.v3.position.y),
                              fminf(fminf(t.v1.position.z, t.v2.position.z), t.v3.position.z) };
        const float hi[3] = { fmaxf(fmaxf(t.v1.position.x, t.v2.position.x), t.v3.position.x), fmaxf(fmaxf(t.v1.position.y, t.v2.position.y), t.v3.position.y),
                              fmaxf(fmaxf(t.v1.position.z, t.v2.position.z), t.v3.position.z) };
        if (!(lo[0] == nd.bmin.x && lo[1] == nd.bmin.y && lo[2] == nd.bmin.z && hi[0] == nd.bmax.x && hi[1] == nd.bmax.y && hi[2] == nd.bmax.z))
            atomicOr(error, REFIT_ERR_LEAF_BOX);
    }
}

__global__ void refit_shade_kernel(ShadeTri* __restrict__ shade, const RefTriangle* __restrict__ tris, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RefTriangle& t = tris[i];
    ShadeTri s;
    s.n1[0] = t.v1.normal.x; s.n1[1] = t.v1.normal.y; s.n1[2] = t.v1.normal.z; s.mtl = t.mtlIndex;
    s.n2[0] = t.v2.normal.x; s.n2[1] = t.v2.normal.y; s.n2[2] = t.v2.normal.z; s.pad0 = 0;
    s.n3[0] = t.v3.normal.x; s.n3[1] = t.v3.normal.y; s.n3[2] = t.v3.normal.z; s.pad1 = 0;
    shade[i] = s;
}

int refit_one(b2rt_context* ctx, const void* triangles, uint64_t n_triangles) {
    int st = use_device(ctx);
    if (st) return st;
    Buffer* bt = find(ctx, ctx->bound[B2RT_ARG_BUFFER_SCENE]);
    Buffer* bn = find(ctx, ctx->bound[B2RT_ARG_BUFFER_NODE]);
    if (!bt || !bn || ctx->scene_dirty || !ctx->d_child_bin) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "refit needs an uploaded, built scene");
    if (n_triangles * sizeof(RefTriangle) != bt->bytes)
        return fail(ctx, B2RT_INVALID_VALUE, "refit: " + std::to_string(n_triangles) + " triangles given, the scene has " + std::to_string(bt->bytes / sizeof(RefTriangle)));
    const uint32_t n_nodes = (uint32_t)ctx->info.n_nodes, n_wide = (uint32_t)ctx->info.n_wide_nodes, n_blocks = (uint32_t)ctx->info.n_leaf_blocks,
                   n_tris = (uint32_t)n_triangles;
    cudaStream_t s = ctx->stream;
    if (triangles) CK(cudaMemcpyAsync(bt->d_ptr, triangles, bt->bytes, cudaMemcpyHostToDevice, s));     // null: the caller wrote the device buffer itself
    char* scratch = nullptr;
    CK(cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)n_nodes * 8 + 256, s));
    int* parent = reinterpret_cast<int*>(scratch);
    unsigned* arrivals = reinterpret_cast<unsigned*>(scratch + (size_t)n_nodes * 4);
    unsigned* error = reinterpret_cast<unsigned*>(scratch + (size_t)n_nodes * 8);
    cudaError_t e = cudaMemsetAsync(error, 0, 4, s);
    RefNode* nodes = static_cast<RefNode*>(bn->d_ptr);
    const RefTriangle* tris = static_cast<const RefTriangle*>(bt->d_ptr);
    auto grid = [](uint32_t n) { return (n + 255u) / 256u; };
    if (e == cudaSuccess) {
        refit_leaf_kernel<<<grid(n_nodes), 256, 0, s>>>(nodes, n_nodes, tris, parent, arrivals);
        refit_up_kernel<<<grid(n_nodes), 256, 0, s>>>(nodes, n_nodes, parent, arrivals);
        refit_wide_kernel<<<grid(n_wide), 256, 0, s>>>(static_cast<WideNode*>(ctx->d_wide), n_wide, ctx->d_child_bin, nodes, error);
        refit_block_kernel<<<grid(n_blocks), 256, 0, s>>>(static_cast<U4*>(ctx->d_leaf), ctx->d_leaf_dir, n_blocks, nodes, tris, error);
        refit_shade_kernel<<<grid(n_tris), 256, 0, s>>>(static_cast<ShadeTri*>(ctx->d_shade), tris, n_tris);
        e = cudaGetLastError();
        ctx->launches += 5;
    }
    unsigned err = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&err, error, 4, cudaMemcpyDeviceToHost, s);
    cudaFreeAsync(scratch, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "refit");
    bt->shadow.clear();
    bn->shadow.clear();
    if (err & REFIT_ERR_NONFINITE) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: non-finite vertex positions; the scene must be uploaded again");
    if (err & REFIT_ERR_RANGE) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: bounds too large to quantise; the scene must be uploaded again");
    if (err & REFIT_ERR_LEAF_BOX) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: a leaf's box is not the min / max of its vertices; the scene must be uploaded again");
    if (err & REFIT_ERR_DUPLICATE)
        return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: two triangles that were the loader's copies of one face no longer are; rebuild the scene instead");
    return B2RT_SUCCESS;
}

int refit_each(b2rt_context* ctx, void* arg) {
    const void* const* a = static_cast<const void* const*>(arg);
    return refit_one(ctx, a[0], *static_cast<const uint64_t*>(a[1]));
}

}  // namespace

namespace b2rt_detail {
cudaError_t launch_shade_records(ShadeTri* shade, const RefTriangle* tris, uint32_t n, cudaStream_t s) {
    if (n) refit_shade_kernel<<<(n + 255u) / 256u, 256, 0, s>>>(shade, tris, n);
    return cudaGetLastError();
}
}  // namespace b2rt_detail

extern "C" int b2rt_refit_scene(b2rt_context* ctx, const void* triangles, uint64_t n_triangles) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!triangles || !n_triangles) return fail(ctx, B2RT_INVALID_VALUE, "refit: null or empty triangle array");
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    if (ctx->group) {                                    // every device refits its own copy
        const void* a[2] = { triangles, &n_triangles };
        return group_each(ctx, refit_each, a, true);
    }
    return refit_one(ctx, triangles, n_triangles);
}
