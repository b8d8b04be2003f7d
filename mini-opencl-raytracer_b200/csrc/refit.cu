// refit.cu -- b2rt_refit_scene / b2rt_refit_scene_device: new vertex data for the bound scene, same topology. Everything
// the kernels read is refreshed ON THE DEVICE, no tree is rebuilt (SURVEY.md 8f-2 "build / refit"; the reference can only
// re-run CLBVHScene::RecursiveBuild, CLBVHnode.cpp:7-159, and upload again). Both entry points enqueue the same sequence
// (refit_load, refit_kernels) on a given stream with a given error word:
//   1. the new CLTriangle array replaces the bound triangle buffer: one H2D copy (host entry), one D2D copy, nothing
//      (the data is already in the bound buffer), or refit_gather_kernel through the build's order (device entry);
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
#include <atomic>
#include <string>
#include "context.h"

using namespace b2rt;
using namespace b2rt_detail;

namespace {

// out[k] = in[order[k]] for the k whose order entry is in range; an entry >= n leaves record k as it was and sets
// B2RT_REFIT_ORDER. Sixteen threads per 256-byte record, one 16-byte word each (scene_build.cu's gather_kernel plus the
// bounds check: a bad order must never become an out-of-bounds read).
__global__ void refit_gather_kernel(const uint4* __restrict__ in, const uint32_t* __restrict__ order, uint32_t n, uint4* __restrict__ out,
                                    unsigned* __restrict__ error) {
    const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= (uint64_t)n * 16) return;
    const uint32_t k = (uint32_t)(w >> 4), l = (uint32_t)(w & 15);
    const uint32_t src = __ldg(order + k);
    if (src >= n) { if (l == 0) atomicOr(error, (unsigned)B2RT_REFIT_ORDER); return; }
    out[w] = __ldg(in + (size_t)src * 16 + l);
}

// finite_error != nullptr: every vertex coordinate is checked too (B2RT_REFIT_NONFINITE). The min / max chain drops a NaN,
// so a NaN that both copies of a loader pair share would otherwise pass unreported.
__global__ void refit_leaf_kernel(RefNode* __restrict__ nodes, uint32_t n_nodes, const RefTriangle* __restrict__ tris, int* __restrict__ parent,
                                  unsigned* __restrict__ arrivals, unsigned* __restrict__ finite_error) {
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
            if (finite_error && !(isfinite(p[k]->x) && isfinite(p[k]->y) && isfinite(p[k]->z))) atomicOr(finite_error, (unsigned)B2RT_REFIT_NONFINITE);
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
        if (!(lo[a] <= hi[a]) || !isfinite(lo[a]) || !isfinite(hi[a])) { atomicOr(error, (unsigned)B2RT_REFIT_NONFINITE); return; }
        wn.base[a] = lo[a];
        int e = 1;
        const double extent = (double)hi[a] - (double)lo[a];
        if (extent > 0.0) { int k; (void)frexp(extent / 255.0, &k); e = min(max(k + 127, 1), 254); }
        for (;; ++e) {
            if (e > 230) { atomicOr(error, (unsigned)B2RT_REFIT_RANGE); return; }
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
            if (!ok) atomicOr(error, (unsigned)B2RT_REFIT_DUPLICATE);
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
            atomicOr(error, (unsigned)B2RT_REFIT_LEAF_BOX);
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

// The bound scene's triangle and node buffers, for a refit with n_triangles triangles.
int refit_target(b2rt_context* ctx, uint64_t n_triangles, Buffer** bt, Buffer** bn) {
    *bt = find(ctx, ctx->bound[B2RT_ARG_BUFFER_SCENE]);
    *bn = find(ctx, ctx->bound[B2RT_ARG_BUFFER_NODE]);
    if (!*bt || !*bn || ctx->scene_dirty || !ctx->d_child_bin) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "refit needs an uploaded, built scene");
    if (n_triangles * sizeof(RefTriangle) != (*bt)->bytes)
        return fail(ctx, B2RT_INVALID_VALUE, "refit: " + std::to_string(n_triangles) + " triangles given, the scene has " + std::to_string((*bt)->bytes / sizeof(RefTriangle)));
    return B2RT_SUCCESS;
}

// Step 1 on stream s: the new scene-order triangles into the bound triangle buffer.
//   src == nullptr or src == the bound buffer   it already holds them: nothing to do
//   order == nullptr                            src holds them: one copy of kind `kind`
//   order != nullptr                            scene triangle k is src[order[k]] (device memory): the gather, which ORs
//                                               B2RT_REFIT_ORDER into *error for an entry out of range
cudaError_t refit_load(b2rt_context* ctx, Buffer* bt, const void* src, cudaMemcpyKind kind, const uint32_t* order, unsigned* error, cudaStream_t s) {
    const uint32_t n_tris = (uint32_t)(bt->bytes / sizeof(RefTriangle));
    if (order) {
        refit_gather_kernel<<<(unsigned)((16ull * n_tris + 255u) / 256u), 256, 0, s>>>(static_cast<const uint4*>(src), order, n_tris, static_cast<uint4*>(bt->d_ptr), error);
        ctx->launches += 1;
        return cudaGetLastError();
    }
    if (src && src != bt->d_ptr) return cudaMemcpyAsync(bt->d_ptr, src, bt->bytes, kind, s);
    return cudaSuccess;
}

// Step 2 on stream s: boxes, wide nodes, leaf blocks and shading records from the bound triangle buffer; error bits are
// ORed into the device word *error. check_finite: every vertex is checked for non-finite coordinates as well (the device
// entry; the host entry keeps the checks it has always made).
cudaError_t refit_kernels(b2rt_context* ctx, Buffer* bt, Buffer* bn, unsigned* error, bool check_finite, cudaStream_t s) {
    const uint32_t n_nodes = (uint32_t)ctx->info.n_nodes, n_wide = (uint32_t)ctx->info.n_wide_nodes, n_blocks = (uint32_t)ctx->info.n_leaf_blocks,
                   n_tris = (uint32_t)(bt->bytes / sizeof(RefTriangle));
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)n_nodes * 8, s);
    if (e != cudaSuccess) return e;
    int* parent = reinterpret_cast<int*>(scratch);
    unsigned* arrivals = reinterpret_cast<unsigned*>(scratch + (size_t)n_nodes * 4);
    RefNode* nodes = static_cast<RefNode*>(bn->d_ptr);
    const RefTriangle* tris = static_cast<const RefTriangle*>(bt->d_ptr);
    auto grid = [](uint32_t n) { return (n + 255u) / 256u; };
    refit_leaf_kernel<<<grid(n_nodes), 256, 0, s>>>(nodes, n_nodes, tris, parent, arrivals, check_finite ? error : nullptr);
    refit_up_kernel<<<grid(n_nodes), 256, 0, s>>>(nodes, n_nodes, parent, arrivals);
    refit_wide_kernel<<<grid(n_wide), 256, 0, s>>>(static_cast<WideNode*>(ctx->d_wide), n_wide, ctx->d_child_bin, nodes, error);
    refit_block_kernel<<<grid(n_blocks), 256, 0, s>>>(static_cast<U4*>(ctx->d_leaf), ctx->d_leaf_dir, n_blocks, nodes, tris, error);
    refit_shade_kernel<<<grid(n_tris), 256, 0, s>>>(static_cast<ShadeTri*>(ctx->d_shade), tris, n_tris);
    e = cudaGetLastError();
    ctx->launches += 5;
    cudaFreeAsync(scratch, s);
    bt->shadow.clear();
    bn->shadow.clear();
    return e;
}

// Refit of this device's bound scene on its own stream, waited for: host triangles (H2D copy), or nullptr when the bound
// buffer already holds the new data. *bits receives the B2RT_REFIT_* bits; check_finite as for refit_kernels.
int refit_sync(b2rt_context* ctx, const void* triangles, uint64_t n_triangles, bool check_finite, unsigned* bits) {
    int st = use_device(ctx);
    if (st) return st;
    Buffer *bt, *bn;
    st = refit_target(ctx, n_triangles, &bt, &bn);
    if (st) return st;
    cudaStream_t s = ctx->stream;
    unsigned* error = nullptr;
    CK(cudaMallocAsync(reinterpret_cast<void**>(&error), 4, s));
    cudaError_t e = cudaMemsetAsync(error, 0, 4, s);
    if (e == cudaSuccess) e = refit_load(ctx, bt, triangles, cudaMemcpyHostToDevice, nullptr, error, s);
    if (e == cudaSuccess) e = refit_kernels(ctx, bt, bn, error, check_finite, s);
    unsigned err = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&err, error, 4, cudaMemcpyDeviceToHost, s);
    cudaFreeAsync(error, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "refit");
    *bits = err;
    return B2RT_SUCCESS;
}

int refit_one(b2rt_context* ctx, const void* triangles, uint64_t n_triangles) {
    unsigned err = 0;
    int st = refit_sync(ctx, triangles, n_triangles, false, &err);
    if (st) return st;
    if (err & B2RT_REFIT_NONFINITE) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: non-finite vertex positions; the scene must be uploaded again");
    if (err & B2RT_REFIT_RANGE) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: bounds too large to quantise; the scene must be uploaded again");
    if (err & B2RT_REFIT_LEAF_BOX) return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: a leaf's box is not the min / max of its vertices; the scene must be uploaded again");
    if (err & B2RT_REFIT_DUPLICATE)
        return fail(ctx, B2RT_INVALID_ARG_VALUE, "refit: two triangles that were the loader's copies of one face no longer are; rebuild the scene instead");
    return B2RT_SUCCESS;
}

int refit_each(b2rt_context* ctx, void* arg) {
    const void* const* a = static_cast<const void* const*>(arg);
    return refit_one(ctx, a[0], *static_cast<const uint64_t*>(a[1]));
}

// Device group, device entry: every member refits the copy of the new triangles it has been given; the bits are ORed.
struct GroupRefit { uint64_t n; std::atomic<unsigned> bits; };
int refit_member(b2rt_context* ctx, void* arg) {
    GroupRefit* g = static_cast<GroupRefit*>(arg);
    unsigned err = 0;
    int st = refit_sync(ctx, nullptr, g->n, true, &err);
    g->bits |= err;
    return st;
}

// B2RT_INVALID_VALUE unless p is device or managed memory of ctx's device.
int check_device_memory(b2rt_context* ctx, const void* p, const char* what) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) { cudaGetLastError(); return fail(ctx, B2RT_INVALID_VALUE, std::string(what) + ": not a CUDA pointer"); }
    if ((attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) || attr.device != ctx->device)
        return fail(ctx, B2RT_INVALID_VALUE, std::string(what) + ": not device memory of device " + std::to_string(ctx->device));
    return B2RT_SUCCESS;
}

bool overlap(const void* a, size_t a_bytes, const void* b, size_t b_bytes) {
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + b_bytes && y < x + a_bytes;
}

}  // namespace

namespace b2rt_detail {
cudaError_t stream_edge(cudaEvent_t ev, cudaStream_t from, cudaStream_t to) {
    cudaError_t e = cudaEventRecord(ev, from);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(to, ev, 0);
    return e;
}
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

extern "C" int b2rt_refit_scene_device(b2rt_context* ctx, const void* d_triangles, uint64_t n_triangles, const uint32_t* d_order, uint32_t* d_status,
                                       void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!d_triangles || !n_triangles) return fail(ctx, B2RT_INVALID_VALUE, "refit: null or empty triangle array");
    if (!d_status) return fail(ctx, B2RT_INVALID_VALUE, "refit: a device status word is required");
    // the kernels read the records with 16-byte loads and the words with 4-byte ones: a misaligned view would fault
    if (reinterpret_cast<uintptr_t>(d_triangles) % 16) return fail(ctx, B2RT_INVALID_VALUE, "triangles: device address is not 16-byte aligned");
    if (reinterpret_cast<uintptr_t>(d_order) % 4) return fail(ctx, B2RT_INVALID_VALUE, "order: device address is not 4-byte aligned");
    if (reinterpret_cast<uintptr_t>(d_status) % 4) return fail(ctx, B2RT_INVALID_VALUE, "status: device address is not 4-byte aligned");
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    Buffer *bt, *bn;
    st = refit_target(ctx, n_triangles, &bt, &bn);
    if (st) return st;
    st = check_device_memory(ctx, d_triangles, "triangles");
    if (!st && d_order) st = check_device_memory(ctx, d_order, "order");
    if (!st) st = check_device_memory(ctx, d_status, "status");
    if (st) return st;
    const size_t bytes = bt->bytes;
    if (overlap(d_triangles, bytes, bt->d_ptr, bytes) && (d_order || d_triangles != bt->d_ptr))
        return fail(ctx, B2RT_INVALID_VALUE, d_order ? "refit: a gather cannot read the bound triangle buffer it writes"
                                                     : "refit: the triangles overlap the bound triangle buffer without being it");
    if (d_order && overlap(d_order, (size_t)n_triangles * 4, bt->d_ptr, bytes))
        return fail(ctx, B2RT_INVALID_VALUE, "refit: the order lies in the bound triangle buffer the gather writes");
    cudaStream_t s = ctx->stream, caller = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : s;
    if (caller != s) CK(stream_edge(ctx->ev_refit[0], caller, s));              // behind the caller's work on its stream
    CK(cudaMemsetAsync(d_status, 0, 4, s));
    if (!ctx->group) {
        CK(refit_load(ctx, bt, d_triangles, cudaMemcpyDefault, d_order, d_status, s));
        CK(refit_kernels(ctx, bt, bn, d_status, true, s));
        if (caller != s) CK(stream_edge(ctx->ev_refit[1], s, caller));          // the caller's later work sees the refitted scene
        return B2RT_SUCCESS;
    }
    // device group: the root puts the new scene-order triangles into its bound buffer, the peers get copies, every member
    // refits its own; synchronous, d_status = OR of every member's bits
    CK(refit_load(ctx, bt, d_triangles, cudaMemcpyDefault, d_order, d_status, s));
    st = group_broadcast_buffer(ctx, ctx->bound[B2RT_ARG_BUFFER_SCENE]);    // waits for every member's stream
    if (st) return st;
    GroupRefit g;
    g.n = n_triangles;
    g.bits = 0u;
    st = group_each(ctx, refit_member, &g, true);
    if (st) return st;
    unsigned bits = 0;
    CK(cudaMemcpyAsync(&bits, d_status, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    bits |= g.bits.load();
    CK(cudaMemcpyAsync(d_status, &bits, 4, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));
    return B2RT_SUCCESS;
}
