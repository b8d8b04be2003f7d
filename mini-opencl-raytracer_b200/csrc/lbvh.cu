// lbvh.cu -- binary BVH build on the device (SURVEY.md 8f-2): a linear BVH (Morton order + Karras 2012) over
// primitive GROUPS, returned to the host in a form that api.cu flattens into the REFERENCE's own
// CLLinearBVHNode array + triangle order, i.e. a drop-in for what CLBVHScene::RecursiveBuild +
// FlattenBVHTree produce (CLBVHnode.cpp:7-183) -- a different tree, same format, same consumers.
//
// A group is a run of consecutive loader triangles with bit-identical centroids: the loader emits every OBJ face
// as 2 (triangle) or 3 (quad) overlapping triangles (CLOBJloader.cpp:102-126) and the reference's builder can never
// separate them (identical centroids), so they stay one leaf here too.
//
//   morton_kernel      30-bit Morton code of each group's centroid inside the scene box
//   radix passes       stable LSD radix sort, 8 bits per pass (4 passes for the 30-bit codes): per-block digit histogram,
//                      one scan of the digit-major block histograms, scatter with warp-match ranking (12 launches; r1 used
//                      one-bit split passes, 90 launches)
//   karras_kernel      one thread per internal node: range, split, children, parent links, split axis
//   refit_kernel       one thread per leaf walks up; the second arrival at a node unions its children's boxes
//   leaf offsets       exclusive scan of the group sizes in Morton order = first triangle of every leaf after re-ordering
//   flatten_kernel     FlattenBVHTree (CLBVHnode.cpp:161-183) without the recursion: a node's pre-order index is the sum,
//                      over its ancestors, of 1 (it is in the first subtree) or 1 + the first subtree's node count (it is
//                      in the second); a Karras node over k leaves has 2k - 1 nodes, so one walk up per node gives its
//                      index, and the CLLinearBVHNode records are written in place. order_kernel lists the triangles leaf
//                      by leaf (what CreateBVHTrees re-orders m_Triangles by, CLBVHnode.cpp:197).
#include <cuda_runtime.h>
#include <stdint.h>
#include "lbvh.h"

namespace b2rt {

namespace {

constexpr int SCAN_BLOCK = 1024;

__device__ __forceinline__ uint32_t expand10(uint32_t v) {      // 10 bits -> every third bit
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void morton_kernel(const float* __restrict__ bounds, uint32_t m, float3 lo, float3 inv, uint32_t* __restrict__ keys,
                              uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float* b = bounds + 6 * (size_t)i;
    float cx = (0.5f * b[0] + 0.5f * b[3] - lo.x) * inv.x, cy = (0.5f * b[1] + 0.5f * b[4] - lo.y) * inv.y,
          cz = (0.5f * b[2] + 0.5f * b[5] - lo.z) * inv.z;
    uint32_t x = (uint32_t)fminf(fmaxf(cx * 1024.0f, 0.0f), 1023.0f), y = (uint32_t)fminf(fmaxf(cy * 1024.0f, 0.0f), 1023.0f),
             z = (uint32_t)fminf(fmaxf(cz * 1024.0f, 0.0f), 1023.0f);
    keys[i] = (expand10(x) << 2) | (expand10(y) << 1) | expand10(z);      // bit b of the code: axis 2 - b % 3
    vals[i] = i;
}

// Radix pass, step 1: digit histogram of each block of SCAN_BLOCK keys, stored digit-major (hist[digit * n_blocks + block])
// so that ONE exclusive scan of the whole array yields every (digit, block) group's first output position.
__global__ void __launch_bounds__(SCAN_BLOCK) radix_hist_kernel(const uint32_t* __restrict__ keys, uint32_t m, uint32_t shift, uint32_t n_blocks,
                                                                 uint32_t* __restrict__ hist) {
    __shared__ uint32_t h[256];
    if (threadIdx.x < 256) h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * SCAN_BLOCK + threadIdx.x;
    if (i < m) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
    __syncthreads();
    if (threadIdx.x < 256) hist[threadIdx.x * n_blocks + blockIdx.x] = h[threadIdx.x];
}

// Radix pass, step 3: stable scatter. Rank of a key among the block's earlier keys with the same digit = (keys of that digit
// in earlier warps) + (earlier lanes of its own warp holding the digit, from __match_any_sync).
__global__ void __launch_bounds__(SCAN_BLOCK) radix_scatter_kernel(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals, uint32_t m,
                                                                    uint32_t shift, uint32_t n_blocks, const uint32_t* __restrict__ offsets,
                                                                    uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out) {
    __shared__ uint16_t count[SCAN_BLOCK / 32][256];          // per warp and digit: keys held, then keys in earlier warps
    for (uint32_t k = threadIdx.x; k < (SCAN_BLOCK / 32) * 256; k += SCAN_BLOCK) (&count[0][0])[k] = 0;
    __syncthreads();
    const uint32_t i = blockIdx.x * SCAN_BLOCK + threadIdx.x, lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t key = i < m ? keys[i] : 0u;
    const uint32_t digit = i < m ? (key >> shift) & 255u : 256u;                // 256: past the end, matches only its like
    const uint32_t peers = __match_any_sync(0xffffffffu, digit);
    const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
    if (digit < 256u && rank == 0u) count[warp][digit] = (uint16_t)__popc(peers);
    __syncthreads();
    if (threadIdx.x < 256) {
        uint32_t run = 0;
        for (int w = 0; w < SCAN_BLOCK / 32; ++w) { const uint32_t c = count[w][threadIdx.x]; count[w][threadIdx.x] = (uint16_t)run; run += c; }
    }
    __syncthreads();
    if (i >= m) return;
    const uint32_t dst = offsets[digit * n_blocks + blockIdx.x] + count[warp][digit] + rank;
    keys_out[dst] = key;
    vals_out[dst] = vals[i];
}

// In-place exclusive scan of up to 2^20 * ... block sums by ONE block (loops over the array); total zeros to sums[n].
__global__ void __launch_bounds__(SCAN_BLOCK) sums_scan_kernel(uint32_t* __restrict__ sums, uint32_t n) {
    __shared__ uint32_t warp_sums[SCAN_BLOCK / 32];
    __shared__ uint32_t carry;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += SCAN_BLOCK) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t x = i < n ? sums[i] : 0u;
        uint32_t v = x;
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= (uint32_t)o) v += t; }
        if (lane == 31) warp_sums[warp] = v;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = warp_sums[lane];
            for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= (uint32_t)o) w += t; }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const uint32_t incl = (warp ? warp_sums[warp - 1] : 0u) + v;
        if (i < n) sums[i] = carry + incl - x;
        __syncthreads();
        if (threadIdx.x == SCAN_BLOCK - 1) carry += incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) sums[n] = carry;
}

// Exclusive scan inside each block of SCAN_BLOCK elements (block totals out) and the matching add-back: with sums_scan_kernel
// in between, an exclusive scan of m values.
__global__ void __launch_bounds__(SCAN_BLOCK) block_scan_kernel(const uint32_t* __restrict__ in, uint32_t m, uint32_t* __restrict__ excl,
                                                                 uint32_t* __restrict__ block_sums) {
    __shared__ uint32_t warp_sums[SCAN_BLOCK / 32];
    const uint32_t i = blockIdx.x * SCAN_BLOCK + threadIdx.x, lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t x = i < m ? in[i] : 0u;
    uint32_t v = x;
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= (uint32_t)o) v += t; }
    if (lane == 31) warp_sums[warp] = v;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
        for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, w, o); if (lane >= (uint32_t)o) w += t; }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t before = (warp ? warp_sums[warp - 1] : 0u) + v - x;
    if (i < m) excl[i] = before;
    if (threadIdx.x == SCAN_BLOCK - 1) block_sums[blockIdx.x] = before + x;
}

// Common-prefix length of sorted keys i and j (index tie-break for equal codes), -1 outside the array.
__device__ __forceinline__ int delta(const uint32_t* keys, int m, int i, int j) {
    if (j < 0 || j >= m) return -1;
    const uint32_t a = keys[i], b = keys[j];
    return a != b ? __clz(a ^ b) : 32 + __clz((uint32_t)i ^ (uint32_t)j);
}

// Karras 2012, one thread per internal node i in [0, m-2]. Child reference: index of an internal node, or ~leaf.
__global__ void karras_kernel(const uint32_t* __restrict__ keys, int m, int2* __restrict__ children, int* __restrict__ parent_internal,
                              int* __restrict__ parent_leaf, uint8_t* __restrict__ axis, uint32_t* __restrict__ n_leaves) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m - 1) return;
    const int d = delta(keys, m, i, i + 1) - delta(keys, m, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = delta(keys, m, i, i - d);
    int lmax = 2;
    while (delta(keys, m, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, m, i, i + (l + t) * d) > dmin) l += t;
    const int j = i + l * d;
    const int dnode = delta(keys, m, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(keys, m, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int gamma = i + s * d + min(d, 0);
    const int lo = min(i, j), hi = max(i, j);
    const int left = (lo == gamma) ? ~gamma : gamma, right = (hi == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    children[i] = make_int2(left, right);
    n_leaves[i] = (uint32_t)(hi - lo + 1);
    if (left >= 0) parent_internal[left] = i; else parent_leaf[~left] = i;
    if (right >= 0) parent_internal[right] = i; else parent_leaf[~right] = i;
    // split axis: the first bit in which the range's first and last code differ (bit b of the code belongs to axis 2 - b % 3)
    const uint32_t x = keys[lo] ^ keys[hi];
    axis[i] = x ? (uint8_t)(2 - (31 - __clz(x)) % 3) : (uint8_t)0;
    if (i == 0) parent_internal[0] = -1;
}

__global__ void refit_kernel(const float* __restrict__ group_bounds, const uint32_t* __restrict__ sorted_group, int m,
                             const int2* __restrict__ children, const int* __restrict__ parent_internal, const int* __restrict__ parent_leaf,
                             float* __restrict__ node_bounds, unsigned int* __restrict__ arrivals) {
    const int leaf = blockIdx.x * blockDim.x + threadIdx.x;
    if (leaf >= m) return;
    int node = parent_leaf[leaf];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&arrivals[node], 1u) == 0u) return;           // the first arrival stops; the second sees both children done
        const int2 c = children[node];
        float b[6];
        for (int side = 0; side < 2; ++side) {
            const int r = side ? c.y : c.x;
            // boxes of internal children were written by other threads of this launch: read them past L1 (__ldcg)
            const float* src = r >= 0 ? node_bounds + 6 * (size_t)r : group_bounds + 6 * (size_t)sorted_group[~r];
            for (int k = 0; k < 3; ++k) {
                const float lo = __ldcg(src + k), hi = __ldcg(src + 3 + k);
                b[k] = side ? fminf(b[k], lo) : lo;
                b[3 + k] = side ? fmaxf(b[3 + k], hi) : hi;
            }
        }
        for (int k = 0; k < 6; ++k) node_bounds[6 * (size_t)node + k] = b[k];
        node = parent_internal[node];
    }
}

// Pre-order index of a node: walk up; every ancestor contributes 1 when we came from its first child, 1 + the first
// subtree's node count when we came from its second (a subtree over k leaves has 2k - 1 nodes).
__device__ __forceinline__ uint32_t preorder_index(int ref, int parent, const int2* __restrict__ children, const int* __restrict__ parent_internal,
                                                   const uint32_t* __restrict__ n_leaves) {
    uint32_t idx = 0;
    while (parent >= 0) {
        const int2 c = children[parent];
        idx += 1u;
        if (c.y == ref) idx += c.x >= 0 ? 2u * n_leaves[c.x] - 1u : 1u;
        ref = parent;
        parent = parent_internal[parent];
    }
    return idx;
}

// FlattenBVHTree on the device: thread t < m - 1 writes internal node t, thread m - 1 + l writes leaf l (Morton position l).
__global__ void flatten_kernel(int m, const int2* __restrict__ children, const int* __restrict__ parent_internal, const int* __restrict__ parent_leaf,
                               const uint32_t* __restrict__ n_leaves, const float* __restrict__ node_bounds, const uint8_t* __restrict__ axis,
                               const float* __restrict__ group_bounds, const uint32_t* __restrict__ sorted_group, const uint32_t* __restrict__ first,
                               const uint32_t* __restrict__ leaf_first_tri, RefNode* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * m - 1) return;
    RefNode nd;
    uint32_t* w = reinterpret_cast<uint32_t*>(&nd);
    for (int k = 0; k < 12; ++k) w[k] = 0u;
    uint32_t idx;
    if (t < m - 1) {
        idx = preorder_index(t, parent_internal[t], children, parent_internal, n_leaves);
        const float* b = node_bounds + 6 * (size_t)t;
        nd.bmin.x = b[0]; nd.bmin.y = b[1]; nd.bmin.z = b[2]; nd.bmax.x = b[3]; nd.bmax.y = b[4]; nd.bmax.z = b[5];
        const int2 c = children[t];
        nd.offset = idx + 1u + (c.x >= 0 ? 2u * n_leaves[c.x] - 1u : 1u);       // the second child follows the whole first subtree
        nd.axis = axis[t];
    } else {
        const int l = t - (m - 1);
        idx = preorder_index(~l, parent_leaf[l], children, parent_internal, n_leaves);
        const uint32_t g = sorted_group[l];
        const float* b = group_bounds + 6 * (size_t)g;
        nd.bmin.x = b[0]; nd.bmin.y = b[1]; nd.bmin.z = b[2]; nd.bmax.x = b[3]; nd.bmax.y = b[4]; nd.bmax.z = b[5];
        nd.offset = leaf_first_tri[l];
        nd.nPrimitives = (uint16_t)(first[g + 1] - first[g]);
    }
    out[idx] = nd;
}

__global__ void group_size_kernel(const uint32_t* __restrict__ sorted_group, const uint32_t* __restrict__ first, uint32_t m, uint32_t* __restrict__ sizes) {
    const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < m) { const uint32_t g = sorted_group[l]; sizes[l] = first[g + 1] - first[g]; }
}

// leaf_first_tri[l] += its block's offset; then the triangles of leaf l, in loader order, become triangles
// leaf_first_tri[l] .. of the re-ordered scene.
__global__ void order_kernel(const uint32_t* __restrict__ sorted_group, const uint32_t* __restrict__ first, uint32_t m, uint32_t* __restrict__ leaf_first_tri,
                             const uint32_t* __restrict__ block_offsets, uint32_t* __restrict__ order) {
    const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= m) return;
    const uint32_t at = leaf_first_tri[l] + block_offsets[l / SCAN_BLOCK];
    leaf_first_tri[l] = at;
    const uint32_t g = sorted_group[l], t0 = first[g], n = first[g + 1] - t0;
    for (uint32_t k = 0; k < n; ++k) order[at + k] = t0 + k;
}

// out[i] += block_offsets[i / SCAN_BLOCK]: the add-back that completes block_scan_kernel + sums_scan_kernel.
__global__ void add_block_offsets_kernel(uint32_t* __restrict__ out, uint32_t m, const uint32_t* __restrict__ block_offsets) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[i] += block_offsets[i / SCAN_BLOCK];
}

}  // namespace

size_t scan_scratch_words(uint32_t m) { return (m + SCAN_BLOCK - 1) / SCAN_BLOCK + 1; }

cudaError_t scan_exclusive(const uint32_t* d_in, uint32_t m, uint32_t* d_out, uint32_t* d_sums, uint64_t* launches, cudaStream_t st) {
    if (m == 0) return cudaMemsetAsync(d_sums, 0, 4, st);
    const uint32_t n_blocks = (m + SCAN_BLOCK - 1) / SCAN_BLOCK;
    block_scan_kernel<<<n_blocks, SCAN_BLOCK, 0, st>>>(d_in, m, d_out, d_sums);
    sums_scan_kernel<<<1, SCAN_BLOCK, 0, st>>>(d_sums, n_blocks);
    add_block_offsets_kernel<<<(m + 255u) / 256u, 256, 0, st>>>(d_out, m, d_sums);
    if (launches) *launches += 3;
    // sums_scan_kernel leaves the total in d_sums[n_blocks]; move it to the front for the caller
    return cudaMemcpyAsync(d_sums, d_sums + n_blocks, 4, cudaMemcpyDeviceToDevice, st);
}

size_t lbvh_scratch_bytes(uint32_t m) {
    const size_t n_blocks = (m + SCAN_BLOCK - 1) / SCAN_BLOCK;
    // keys x2, vals x2 (the second pair is reused for leaf sizes / offsets), digit-major block histograms (+1), block sums of
    // the leaf-offset scan (+1), parents (internal + leaf), arrivals, leaf counts, children, node boxes, split axes
    return (size_t)m * 4 * 4 + (256 * n_blocks + 1) * 4 + (n_blocks + 1) * 4 + (size_t)m * 4 * 4 + (size_t)m * sizeof(int2) + (size_t)m * 24 + m + 1024;
}

cudaError_t lbvh_build(const float* d_group_bounds, const uint32_t* d_first, uint32_t m, const float scene_lo[3], const float scene_hi[3],
                       void* d_scratch, RefNode* d_nodes, uint32_t* d_order, uint64_t* launches, cudaStream_t st) {
    if (m < 2) return cudaErrorInvalidValue;
    const uint32_t n_blocks = (m + SCAN_BLOCK - 1) / SCAN_BLOCK;
    uint32_t* p = static_cast<uint32_t*>(d_scratch);
    uint32_t *keys[2] = { p, p + m }, *vals[2] = { p + 2 * (size_t)m, p + 3 * (size_t)m };
    uint32_t* hist = p + 4 * (size_t)m;                               // 256 * n_blocks + 1
    uint32_t* sums = hist + 256 * (size_t)n_blocks + 1;               // n_blocks + 1
    int* parent_internal = reinterpret_cast<int*>(sums + n_blocks + 1);
    int* parent_leaf = parent_internal + m;
    unsigned int* arrivals = reinterpret_cast<unsigned int*>(parent_leaf + m);
    uint32_t* n_leaves = arrivals + m;
    int2* children = reinterpret_cast<int2*>(n_leaves + m + (((size_t)(n_leaves + m) & 7) ? 1 : 0));
    float* node_bounds = reinterpret_cast<float*>(children + m);
    uint8_t* axis = reinterpret_cast<uint8_t*>(node_bounds + 6 * (size_t)m);
    float3 lo = make_float3(scene_lo[0], scene_lo[1], scene_lo[2]);
    float3 inv = make_float3(scene_hi[0] > scene_lo[0] ? 1.0f / (scene_hi[0] - scene_lo[0]) : 0.0f,
                             scene_hi[1] > scene_lo[1] ? 1.0f / (scene_hi[1] - scene_lo[1]) : 0.0f,
                             scene_hi[2] > scene_lo[2] ? 1.0f / (scene_hi[2] - scene_lo[2]) : 0.0f);
    const unsigned g256 = (m + 255u) / 256u;
    morton_kernel<<<g256, 256, 0, st>>>(d_group_bounds, m, lo, inv, keys[0], vals[0]);
    int cur = 0;
    for (uint32_t shift = 0; shift < 30; shift += 8) {
        radix_hist_kernel<<<n_blocks, SCAN_BLOCK, 0, st>>>(keys[cur], m, shift, n_blocks, hist);
        sums_scan_kernel<<<1, SCAN_BLOCK, 0, st>>>(hist, 256u * n_blocks);
        radix_scatter_kernel<<<n_blocks, SCAN_BLOCK, 0, st>>>(keys[cur], vals[cur], m, shift, n_blocks, hist, keys[cur ^ 1], vals[cur ^ 1]);
        cur ^= 1;
    }
    const uint32_t* sorted_group = vals[cur];
    uint32_t* leaf_first_tri = vals[cur ^ 1];                         // free after the last pass
    uint32_t* sizes = keys[cur ^ 1];
    cudaError_t e = cudaMemsetAsync(arrivals, 0, (size_t)m * 4, st);
    if (e != cudaSuccess) return e;
    karras_kernel<<<(m - 1 + 255u) / 256u, 256, 0, st>>>(keys[cur], (int)m, children, parent_internal, parent_leaf, axis, n_leaves);
    refit_kernel<<<g256, 256, 0, st>>>(d_group_bounds, sorted_group, (int)m, children, parent_internal, parent_leaf, node_bounds, arrivals);
    // first triangle of every leaf in the re-ordered scene: exclusive scan of the group sizes in Morton order
    group_size_kernel<<<g256, 256, 0, st>>>(sorted_group, d_first, m, sizes);
    block_scan_kernel<<<n_blocks, SCAN_BLOCK, 0, st>>>(sizes, m, leaf_first_tri, sums);
    sums_scan_kernel<<<1, SCAN_BLOCK, 0, st>>>(sums, n_blocks);
    order_kernel<<<g256, 256, 0, st>>>(sorted_group, d_first, m, leaf_first_tri, sums, d_order);
    flatten_kernel<<<(2u * m - 1u + 255u) / 256u, 256, 0, st>>>((int)m, children, parent_internal, parent_leaf, n_leaves, node_bounds, axis,
                                                               d_group_bounds, sorted_group, d_first, leaf_first_tri, d_nodes);
    if (launches) *launches += 1 + 4 * 3 + 2 + 5;
    return cudaGetLastError();
}

}  // namespace b2rt
