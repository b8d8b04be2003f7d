// scene_build.cu -- b2rt_build_scene_device: a whole scene built on the device from loader-order CLTriangles that are
// already in device memory. Nothing of the scene crosses PCIe; the host only learns sizes (one small read-back after
// grouping, one per wide-BVH level).
//
//   1. grouping      group_flag_kernel / run_cap_kernel / scatter_first_kernel / group_box_kernel: the groups of
//                    b2rt_build_bvh's host pass (runs of bit-identical centroids, cut at every 65536th triangle and
//                    every 255 triangles of a run), so that lbvh_build produces the byte-identical tree
//   2. binary BVH    lbvh_build (lbvh.cu), written straight into the new node buffer
//   3. re-ordering   gather_kernel: 256-byte records, one 16-byte load per thread
//   4. wide BVH      the derivation of wide_bvh.cpp, byte for byte:
//                      plan_init_kernel / plan_up_kernel   plan_cuts bottom-up (second arrival at a node computes it)
//                      level_count_kernel                  per wide node of one level: treelet, child and leaf-word counts
//                      (three scans)                       child_base / leaf_base / leaf-block numbers in FIFO order
//                      level_emit_kernel                   wide nodes, leaf blocks, leaf_dir, child_bin, the next level
//                      need_kernel                         the exact stack bound, levels bottom-up
//                    shading records: refit.cu's kernel
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>
#include "context.h"
#include "lbvh.h"

using namespace b2rt;
using namespace b2rt_detail;

namespace {

enum : unsigned { SB_ERR_VERTEX = 1u, SB_ERR_BOUNDS = 2u, SB_ERR_RANGE = 4u };

constexpr uint32_t GROUP_CHUNK = 1u << 16;   // b2rt_build_bvh's host chunk: a group never straddles a multiple of it
constexpr uint32_t GROUP_CAP = 255;          // ... and holds at most 255 triangles (nPrimitives of a leaf stays small)

// std::min / std::max exactly as the host evaluates them: for equal values (+0 / -0) the same operand wins
__device__ __forceinline__ float hmin(float a, float b) { return b < a ? b : a; }
__device__ __forceinline__ float hmax(float a, float b) { return a < b ? b : a; }

// float -> unsigned with the same order (atomicMin / atomicMax on floats)
__device__ __forceinline__ unsigned ordered(float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }

__device__ __forceinline__ void tri_box(const RefTriangle& t, float lo[3], float hi[3]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(&t.v1.position)), b = __ldg(reinterpret_cast<const float4*>(&t.v2.position)),
                 c = __ldg(reinterpret_cast<const float4*>(&t.v3.position));
    lo[0] = hmin(a.x, hmin(b.x, c.x)); lo[1] = hmin(a.y, hmin(b.y, c.y)); lo[2] = hmin(a.z, hmin(b.z, c.z));
    hi[0] = hmax(a.x, hmax(b.x, c.x)); hi[1] = hmax(a.y, hmax(b.y, c.y)); hi[2] = hmax(a.z, hmax(b.z, c.z));
}

// CLBVHnode.cpp:190-193, the host's operation order: lo * 0.5f + hi * 0.5f, no fused multiply-add
__device__ __forceinline__ void centroid(const RefTriangle& t, uint32_t c[3]) {
    float lo[3], hi[3];
    tri_box(t, lo, hi);
    for (int k = 0; k < 3; ++k) c[k] = __float_as_uint(__fadd_rn(__fmul_rn(lo[k], 0.5f), __fmul_rn(hi[k], 0.5f)));
}

// flag[i] = 1 where a triangle starts a run of equal centroids (or a host chunk); non-finite vertices are reported;
// the scene's centroid box is the min / max over the run starts.
__global__ void group_flag_kernel(const RefTriangle* __restrict__ tris, uint32_t n, uint32_t* __restrict__ flag, unsigned* __restrict__ cbox,
                                  unsigned* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RefTriangle& t = tris[i];
    const float* p[3] = { &t.v1.position.x, &t.v2.position.x, &t.v3.position.x };
    bool finite = true;
    for (int v = 0; v < 3; ++v) for (int k = 0; k < 3; ++k) finite = finite && isfinite(__ldg(p[v] + k));
    if (!finite) atomicOr(error, SB_ERR_VERTEX);
    uint32_t c[3];
    centroid(t, c);
    bool start = i % GROUP_CHUNK == 0;
    if (!start) {
        uint32_t q[3];
        centroid(tris[i - 1], q);
        start = c[0] != q[0] || c[1] != q[1] || c[2] != q[2];
    }
    flag[i] = start ? 1u : 0u;
    if (start)
        for (int k = 0; k < 3; ++k) { atomicMin(cbox + k, ordered(__uint_as_float(c[k]))); atomicMax(cbox + 3 + k, ordered(__uint_as_float(c[k]))); }
}

// The host's `i - first >= 255` cap: inside a run, every 255th triangle starts a group. One thread per run walks it (the
// loader's runs are 2-3 triangles; a run ends at the next chunk cut at the latest).
// Threads of this launch read flag[] entries that others write. That race is benign, and edits must keep it so: a walker
// writes only inside its own run, at start + 255k, and stops at the first set flag, which is the next run's start (set by
// group_flag_kernel before this launch). A thread that sees a cap flag written under it walks from start + 255k and writes
// exactly the positions the run's walker writes; every write stores the same 1.
__global__ void run_cap_kernel(uint32_t* __restrict__ flag, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !flag[i]) return;
    for (uint32_t j = i + 1, k = 1; j < n && !flag[j]; ++j, ++k)
        if (k == GROUP_CAP) { flag[j] = 1u; k = 0; }
}

__global__ void scatter_first_kernel(const uint32_t* __restrict__ flag, const uint32_t* __restrict__ group, uint32_t n, const uint32_t* __restrict__ total,
                                     uint32_t* __restrict__ first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (flag[i]) first[group[i]] = i;
    if (i == 0) first[*total] = n;
}

// Group boxes in the host's order: the first triangle's box, then min / max with each further one.
__global__ void group_box_kernel(const RefTriangle* __restrict__ tris, const uint32_t* __restrict__ first, uint32_t m, float* __restrict__ gb) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= m) return;
    const uint32_t t0 = first[g], t1 = first[g + 1];
    float lo[3], hi[3];
    tri_box(tris[t0], lo, hi);
    for (uint32_t t = t0 + 1; t < t1; ++t) {
        float l[3], h[3];
        tri_box(tris[t], l, h);
        for (int k = 0; k < 3; ++k) { lo[k] = hmin(lo[k], l[k]); hi[k] = hmax(hi[k], h[k]); }
    }
    float* o = gb + 6 * (size_t)g;
    for (int k = 0; k < 3; ++k) { o[k] = lo[k]; o[3 + k] = hi[k]; }
}

// out[k] = in[order[k]]: sixteen threads per 256-byte record, one 16-byte word each
__global__ void gather_kernel(const uint4* __restrict__ in, const uint32_t* __restrict__ order, uint32_t n, uint4* __restrict__ out) {
    const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= (uint64_t)n * 16) return;
    const uint32_t k = (uint32_t)(w >> 4), l = (uint32_t)(w & 15);
    out[w] = __ldg(in + (size_t)__ldg(order + k) * 16 + l);
}

// ---- plan_cuts (wide_bvh.cpp) bottom-up -------------------------------------------------------------------------------
__global__ void plan_init_kernel(const RefNode* __restrict__ nodes, uint32_t n_nodes, int* __restrict__ parent, unsigned* __restrict__ arrivals,
                                 float* __restrict__ dist, uint8_t* __restrict__ split, uint8_t* __restrict__ open_root) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    arrivals[i] = 0u;
    if (i == 0) parent[0] = -1;
    const RefNode& nd = nodes[i];
    if (nd.nPrimitives == 0) { parent[i + 1] = (int)i; parent[nd.offset] = (int)i; return; }
    for (int k = 0; k < 8; ++k) { dist[8 * (size_t)i + k] = 0.0f; split[8 * (size_t)i + k] = 0; }
    open_root[i] = 0;
}

__global__ void plan_up_kernel(const RefNode* __restrict__ nodes, uint32_t n_nodes, const int* __restrict__ parent, unsigned* __restrict__ arrivals,
                               float* __restrict__ dist, uint8_t* __restrict__ split, uint8_t* __restrict__ open_root) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes || nodes[i].nPrimitives == 0) return;
    int node = parent[i];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&arrivals[node], 1u) == 0u) return;          // the second arrival sees both children's rows
        const RefNode& n = nodes[node];
        // children's rows were written by other threads of this launch: read them past L1
        float a[8], b[8];
        for (int k = 0; k < 8; ++k) { a[k] = __ldcg(dist + 8 * (size_t)(node + 1) + k); b[k] = __ldcg(dist + 8 * (size_t)n.offset + k); }
        const float dx = __fsub_rn(n.bmax.x, n.bmin.x), dy = __fsub_rn(n.bmax.y, n.bmin.y), dz = __fsub_rn(n.bmax.z, n.bmin.z);
        float area = __fadd_rn(__fadd_rn(__fmul_rn(dx, dy), __fmul_rn(dx, dz)), __fmul_rn(dy, dz));
        if (!(area >= 0.0f)) area = 0.0f;
        float open_cost[9];
        uint8_t open_split[9];
        for (uint32_t k = 2; k <= 8; ++k) {
            float best = INFINITY;
            uint8_t arg = 1;
            for (uint32_t s = 1; s < k; ++s) {
                const float c = __fadd_rn(a[s - 1], b[k - s - 1]);
                if (c < best) { best = c; arg = (uint8_t)s; }
            }
            open_cost[k] = best;
            open_split[k] = arg;
        }
        float d[8];
        uint8_t sp[8];
        d[0] = __fadd_rn(area, open_cost[8]);
        sp[0] = 0;
        for (uint32_t k = 2; k <= 8; ++k) {
            if (open_cost[k] < d[k - 2]) { d[k - 1] = open_cost[k]; sp[k - 1] = open_split[k]; }
            else { d[k - 1] = d[k - 2]; sp[k - 1] = sp[k - 2]; }
        }
        for (int k = 0; k < 8; ++k) { dist[8 * (size_t)node + k] = d[k]; split[8 * (size_t)node + k] = sp[k]; }
        open_root[node] = open_split[8];
        node = parent[node];
    }
}

// ---- treelets ----------------------------------------------------------------------------------------------------------
struct Treelet {
    int n_t, n_slots;
    int8_t left[15], right[15], slot[15];
    uint8_t axis[15];
    uint32_t bin[15], depth[15];
    uint32_t slot_bin[8], slot_depth[8];
    uint32_t slot_leaf;               // bit c: slot c is a binary leaf
};

// wide_bvh.cpp's cut of the treelet under binary node `bin`, slot numbering (depth first, first child first) included
__device__ void form_treelet(const RefNode* __restrict__ nodes, const uint8_t* __restrict__ split, const uint8_t* __restrict__ open_root, uint32_t bin,
                             uint32_t depth, Treelet& T) {
    T.n_t = 1;
    T.bin[0] = bin; T.depth[0] = depth; T.left[0] = T.right[0] = -1; T.axis[0] = 0;
    if (nodes[bin].nPrimitives == 0) {
        int8_t todo_t[16];
        uint8_t todo_s[16];
        int n_todo = 0;
        todo_t[n_todo] = 0; todo_s[n_todo++] = 8;
        bool root = true;
        while (n_todo) {
            --n_todo;
            const int o = todo_t[n_todo];
            const uint32_t slots = todo_s[n_todo];
            const RefNode& n = nodes[T.bin[o]];
            if (n.nPrimitives > 0) continue;                                  // binary leaf: a leaf slot
            const uint32_t give_first = root ? open_root[T.bin[o]] : split[8 * (size_t)T.bin[o] + (slots - 1)];
            root = false;
            if (give_first == 0) continue;                                    // stays closed: becomes its own wide node
            const int l = T.n_t, r = T.n_t + 1;
            T.axis[o] = n.axis;
            T.left[o] = (int8_t)l; T.right[o] = (int8_t)r;
            T.bin[l] = T.bin[o] + 1u; T.depth[l] = T.depth[o] + 1u; T.left[l] = T.right[l] = -1; T.axis[l] = 0;
            T.bin[r] = n.offset; T.depth[r] = T.depth[o] + 1u; T.left[r] = T.right[r] = -1; T.axis[r] = 0;
            todo_t[n_todo] = (int8_t)l; todo_s[n_todo++] = (uint8_t)give_first;
            todo_t[n_todo] = (int8_t)r; todo_s[n_todo++] = (uint8_t)(slots - give_first);
            T.n_t += 2;
        }
    }
    // slots: terminals in depth-first order, first child first (number_slots without the recursion)
    int8_t stack[16];
    int sp = 0, next = 0;
    stack[sp++] = 0;
    T.slot_leaf = 0;
    while (sp) {
        const int i = stack[--sp];
        if (T.left[i] < 0) {
            T.slot[i] = (int8_t)next;
            T.slot_bin[next] = T.bin[i];
            T.slot_depth[next] = T.depth[i];
            if (nodes[T.bin[i]].nPrimitives > 0) T.slot_leaf |= 1u << next;
            ++next;
            continue;
        }
        stack[sp++] = T.right[i];
        stack[sp++] = T.left[i];
    }
    T.n_slots = next;
}

// visit_order of wide_bvh.cpp for sign octant `oct`: second child first where the ray is negative on the split axis
__device__ uint32_t visit_word(const Treelet& T, uint32_t oct) {
    int8_t stack[16];
    int sp = 0, rank = 0;
    uint32_t word = 0;
    stack[sp++] = 0;
    while (sp) {
        const int i = stack[--sp];
        if (T.left[i] < 0) { word |= (uint32_t)T.slot[i] << (4 * rank++); continue; }
        const bool flip = (oct >> T.axis[i]) & 1u;
        stack[sp++] = flip ? T.left[i] : T.right[i];
        stack[sp++] = flip ? T.right[i] : T.left[i];
    }
    for (; rank < 8; ++rank) word |= 7u << (4 * rank);
    return word;
}

__device__ __forceinline__ bool same_pos(const RefVec& a, const RefVec& b) {
    return __float_as_uint(a.x) == __float_as_uint(b.x) && __float_as_uint(a.y) == __float_as_uint(b.y) && __float_as_uint(a.z) == __float_as_uint(b.z);
}

// emit_leaf's record flags for the record that starts at triangle i of a leaf ending at `end`
__device__ __forceinline__ uint32_t record_flags(const RefTriangle* __restrict__ tris, uint32_t i, uint32_t end) {
    if (i + 1 >= end) return REC_SINGLE;
    const RefTriangle &t = tris[i], &s = tris[i + 1];
    if (same_pos(s.v1.position, t.v2.position) && same_pos(s.v2.position, t.v3.position) && same_pos(s.v3.position, t.v1.position)) return REC_ROT_LEFT;
    if (same_pos(s.v1.position, t.v3.position) && same_pos(s.v2.position, t.v1.position) && same_pos(s.v3.position, t.v2.position)) return REC_ROT_RIGHT;
    return REC_SINGLE;
}

// Records of binary leaf n and whether its box is implied by its one record (emit_leaf)
__device__ uint32_t leaf_records(const RefNode& n, const RefTriangle* __restrict__ tris, bool* implied) {
    const uint32_t end = n.offset + n.nPrimitives;
    uint32_t nrec = 0;
    for (uint32_t i = n.offset; i < end; ++nrec) i += record_flags(tris, i, end) ? 2u : 1u;
    bool imp = nrec == 1;
    if (imp) {
        const RefTriangle& t = tris[n.offset];
        const float* a = &t.v1.position.x; const float* b = &t.v2.position.x; const float* c = &t.v3.position.x;
        const float* lo = &n.bmin.x; const float* hi = &n.bmax.x;
        for (int k = 0; k < 3 && imp; ++k) {
            if (isnan(a[k]) || isnan(b[k]) || isnan(c[k])) imp = false;
            else imp = fminf(fminf(a[k], b[k]), c[k]) == lo[k] && fmaxf(fmaxf(a[k], b[k]), c[k]) == hi[k];
        }
    }
    *implied = imp;
    return nrec;
}

// ---- quantisation exactly as wide_bvh.cpp's long double arithmetic (x87: 64-bit significand, nearest even) ------------
// This is the host derivation's arithmetic on x86-64, where long double is the x87 extended format. On a host whose long
// double is something else (IEEE binary128 on aarch64) the two derivations can differ by one grid step wherever a rounded
// difference lands on the other side of a grid plane or of a power of two. Both grids are conservative (child boxes are
// rounded outward, with one step given away wherever the difference may have been rounded), so traversal results do not
// depend on which one is used; only byte identity of the derived arrays does.
struct LongDouble { bool neg; unsigned long long m; int e; };   // (-1)^neg * m * 2^e

__device__ __forceinline__ void float_parts(float f, uint32_t& mant, int& e) {
    const uint32_t u = __float_as_uint(f) & 0x7fffffffu, ex = u >> 23, fr = u & 0x7fffffu;
    if (ex == 0) { mant = fr; e = -149; } else { mant = fr | 0x800000u; e = (int)ex - 150; }
}

__device__ __forceinline__ int bit_length(unsigned __int128 x) {
    const unsigned long long hi = (unsigned long long)(x >> 64), lo = (unsigned long long)x;
    return hi ? 128 - __clzll((long long)hi) : (lo ? 64 - __clzll((long long)lo) : 0);
}

// Round a positive integer x * 2^e to 64 significant bits, nearest even.
__device__ LongDouble round64(bool neg, unsigned __int128 x, int e) {
    const int nb = bit_length(x);
    if (nb <= 64) return LongDouble{ neg, (unsigned long long)x, e };
    int sh = nb - 64;
    unsigned __int128 q = x >> sh;
    const unsigned __int128 rem = x & ((((unsigned __int128)1) << sh) - 1), half = ((unsigned __int128)1) << (sh - 1);
    if (rem > half || (rem == half && (q & 1))) { q += 1; if (q >> 64) { q >>= 1; ++sh; } }
    return LongDouble{ neg, (unsigned long long)q, e + sh };
}

// (long double)a - (long double)b: the exact difference, rounded once. The difference of two floats whose exponents lie
// more than 100 apart is the larger operand to 64 bits (the smaller one is below half an ulp).
__device__ LongDouble ld_sub(float a, float b) {
    uint32_t ma, mb;
    int ea, eb;
    float_parts(a, ma, ea);
    float_parts(b, mb, eb);
    const bool na = __float_as_uint(a) >> 31, nb = !(__float_as_uint(b) >> 31);      // a + (-b)
    if (ma == 0 && mb == 0) return LongDouble{ false, 0ull, 0 };
    if (mb == 0) return LongDouble{ na, ma, ea };
    if (ma == 0) return LongDouble{ nb, mb, eb };
    const int emin = min(ea, eb);
    if (ea - emin > 100) return LongDouble{ na, ma, ea };
    if (eb - emin > 100) return LongDouble{ nb, mb, eb };
    const unsigned __int128 A = ((unsigned __int128)ma) << (ea - emin), B = ((unsigned __int128)mb) << (eb - emin);
    if (na == nb) return round64(na, A + B, emin);
    if (A == B) return LongDouble{ false, 0ull, 0 };
    return A > B ? round64(na, A - B, emin) : round64(nb, B - A, emin);
}

// frexp exponent of (double)(((long double)hi - (long double)lo) / 255.0L) for hi > lo: the grid's start exponent
__device__ int extent_exponent(float hi, float lo) {
    const LongDouble d = ld_sub(hi, lo);
    const int z = __clzll((long long)d.m);
    const unsigned long long m = d.m << z;                       // value = m * 2^(e), m in [2^63, 2^64)
    const int e = d.e - z;
    const unsigned __int128 N = ((unsigned __int128)m) << 64;    // value / 255 = (Q + r / 255) * 2^(e - 64)
    const unsigned __int128 Q = N / 255u;
    const unsigned r = (unsigned)(N % 255u);
    int sh = bit_length(Q) - 64;
    unsigned __int128 q = Q >> sh;
    const unsigned __int128 rem = Q & ((((unsigned __int128)1) << sh) - 1), half = ((unsigned __int128)1) << (sh - 1);
    if (rem > half || (rem == half && (r != 0 || (q & 1)))) { q += 1; if (q >> 64) { q >>= 1; ++sh; } }
    // long double -> double: 64 -> 53 bits, nearest even
    unsigned long long q53 = (unsigned long long)q >> 11;
    const unsigned long long rem2 = (unsigned long long)q & 0x7ffull;
    int carry = 0;
    if (rem2 > 0x400ull || (rem2 == 0x400ull && (q53 & 1ull))) { ++q53; if (q53 >> 53) { q53 >>= 1; carry = 1; } }
    return 53 + (e - 64 + sh + 11 + carry);                      // q53 in [2^52, 2^53)
}

__device__ __forceinline__ int float_ilogb(float f) {
    const uint32_t u = __float_as_uint(f) & 0x7fffffffu, ex = u >> 23;
    return ex ? (int)ex - 127 : (31 - __clz((int)(u & 0x7fffffu))) - 149;
}

// floor and ceil of m * 2^sh, both capped at 4096 (enough for the clamps below)
__device__ __forceinline__ void scaled_floor_ceil(unsigned long long m, int sh, long long& fl, long long& ce) {
    if (m == 0) { fl = ce = 0; return; }
    if (sh >= 0) { fl = ce = (sh >= 13 || m > (4096ull >> sh)) ? 4096 : (long long)(m << sh); return; }
    const int k = -sh;
    if (k >= 64) { fl = 0; ce = 1; return; }
    const unsigned long long f = m >> k;
    const bool frac = (m & ((1ull << k) - 1ull)) != 0;
    fl = f > 4096ull ? 4096 : (long long)f;
    ce = f >= 4096ull ? 4096 : (long long)f + (frac ? 1 : 0);
}

__device__ __forceinline__ bool far_apart(float x, float base) {
    return x != 0.0f && base != 0.0f && abs(float_ilogb(x) - float_ilogb(base)) > 36;
}

// quant_floor / quant_ceil of wide_bvh.cpp with the step s = 2^p: ((long double)x - base) / s is exact up to the
// one rounding of the difference, which ld_sub reproduces.
__device__ int quant_floor_x(float base, int p, float lo) {
    const LongDouble d = ld_sub(lo, base);
    long long fl, ce;
    scaled_floor_ceil(d.m, d.e - p, fl, ce);
    long long q = d.neg ? -ce : fl;
    if (far_apart(lo, base)) q -= 1;
    return (int)min(max(q, 0ll), 255ll);
}
__device__ int quant_ceil_x(float base, int p, float hi) {
    const LongDouble d = ld_sub(hi, base);
    long long fl, ce;
    scaled_floor_ceil(d.m, d.e - p, fl, ce);
    long long q = d.neg ? -fl : ce;
    if (far_apart(hi, base)) q += 1;
    return (int)min(max(q, 0ll), 1000ll);
}

// ---- one level of the wide BVH ----------------------------------------------------------------------------------------
// Per wide node: interior children (treelet terminals that are binary interior nodes, plus leaves whose block would lie
// beyond META_MAX_LEAF_OFFSET), 16-byte leaf words and leaf blocks it emits.
__global__ void level_count_kernel(const uint2* __restrict__ items, uint32_t n_items, const RefNode* __restrict__ nodes, const RefTriangle* __restrict__ tris,
                                   const uint8_t* __restrict__ split, const uint8_t* __restrict__ open_root, uint32_t* __restrict__ n_interior,
                                   uint32_t* __restrict__ n_words, uint32_t* __restrict__ n_blocks) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    Treelet T;
    const uint2 it = items[i];
    form_treelet(nodes, split, open_root, it.x, it.y, T);
    uint32_t rel = 0, interior = 0, blocks = 0;
    for (int c = 0; c < T.n_slots; ++c) {
        if (!((T.slot_leaf >> c) & 1u) || (rel > META_MAX_LEAF_OFFSET && T.n_slots > 1)) { ++interior; continue; }
        bool implied;
        const uint32_t nrec = leaf_records(nodes[T.slot_bin[c]], tris, &implied);
        rel += LEAF_RECORD_WORDS * nrec + (implied ? 0u : (uint32_t)LEAF_BOX_WORDS);
        ++blocks;
    }
    n_interior[i] = interior;
    n_words[i] = rel;
    n_blocks[i] = blocks;
}

struct LevelBases { uint32_t first_wide, child_base, leaf_base, block_base; };

__global__ void level_emit_kernel(const uint2* __restrict__ items, uint32_t n_items, LevelBases lb, const RefNode* __restrict__ nodes,
                                  const RefTriangle* __restrict__ tris, const uint8_t* __restrict__ split, const uint8_t* __restrict__ open_root,
                                  const uint32_t* __restrict__ interior_before, const uint32_t* __restrict__ words_before,
                                  const uint32_t* __restrict__ blocks_before, WideNode* __restrict__ wide, U4* __restrict__ leaf,
                                  uint32_t* __restrict__ leaf_dir, uint32_t* __restrict__ child_bin, uint2* __restrict__ next_items,
                                  unsigned* __restrict__ max_depth_binary, unsigned* __restrict__ error) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    Treelet T;
    const uint2 it = items[i];
    form_treelet(nodes, split, open_root, it.x, it.y, T);
    const uint32_t w = lb.first_wide + i, leaf_base = lb.leaf_base + words_before[i], child_base = lb.child_base + interior_before[i];
    uint32_t block = lb.block_base + blocks_before[i];
    uint32_t deepest = 0;
    for (int k = 0; k < T.n_t; ++k) deepest = max(deepest, T.depth[k]);
    atomicMax(max_depth_binary, deepest);
    WideNode wn;
    memset(&wn, 0, sizeof(wn));
    const int nc = T.n_slots;
    wn.n_children = (uint8_t)nc;
    wn.leaf_base = leaf_base;
    wn.child_base = child_base;

    // children: leaf blocks first (slot order), then the interior references -- and the next level's work items, written
    // before anything here can fail so that the next level never reads an unset item
    uint32_t rel = 0, wrap = 0;
    for (int c = 0; c < nc; ++c) {
        if (!((T.slot_leaf >> c) & 1u)) continue;
        if (rel > META_MAX_LEAF_OFFSET && nc > 1) { wrap |= 1u << c; continue; }
        wn.meta[c] = (uint8_t)rel;
        const RefNode& n = nodes[T.slot_bin[c]];
        bool implied;
        const uint32_t nrec = leaf_records(n, tris, &implied);
        U4* p = leaf + leaf_base + rel;
        leaf_dir[2 * (size_t)block] = T.slot_bin[c];
        leaf_dir[2 * (size_t)block + 1] = leaf_base + rel;
        ++block;
        const uint32_t end = n.offset + n.nPrimitives;
        uint32_t k = 0;
        for (uint32_t t = n.offset; t < end; ++k) {
            const uint32_t flags = record_flags(tris, t, end);
            const RefTriangle& tr = tris[t];
            const uint32_t w0 = flags | (k == 0 ? (nrec << LEAF_NREC_SHIFT) | (implied ? 0u : LEAF_HAS_BOX) : 0u);
            p[3 * k + 0] = U4{ __float_as_uint(tr.v1.position.x), __float_as_uint(tr.v1.position.y), __float_as_uint(tr.v1.position.z), w0 };
            p[3 * k + 1] = U4{ __float_as_uint(tr.v2.position.x), __float_as_uint(tr.v2.position.y), __float_as_uint(tr.v2.position.z), k == 0 ? n.offset : 0u };
            p[3 * k + 2] = U4{ __float_as_uint(tr.v3.position.x), __float_as_uint(tr.v3.position.y), __float_as_uint(tr.v3.position.z), 0u };
            t += flags ? 2u : 1u;
        }
        rel += LEAF_RECORD_WORDS * nrec;
        if (!implied) {
            p[3 * nrec + 0] = U4{ __float_as_uint(n.bmin.x), __float_as_uint(n.bmin.y), __float_as_uint(n.bmin.z), 0u };
            p[3 * nrec + 1] = U4{ __float_as_uint(n.bmax.x), __float_as_uint(n.bmax.y), __float_as_uint(n.bmax.z), 0u };
            rel += LEAF_BOX_WORDS;
        }
    }
    uint32_t n_int = 0;
    for (int c = 0; c < nc; ++c) {
        if (((T.slot_leaf >> c) & 1u) && !((wrap >> c) & 1u)) continue;
        wn.meta[c] = (uint8_t)(META_INTERIOR | n_int);
        next_items[interior_before[i] + n_int] = make_uint2(T.slot_bin[c], T.slot_depth[c]);
        ++n_int;
    }
    for (int c = 0; c < 8; ++c) child_bin[8 * (size_t)w + c] = c < nc ? T.slot_bin[c] : 0xFFFFFFFFu;

    // quantisation frame
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int c = 0; c < nc; ++c) {
        const RefNode& n = nodes[T.slot_bin[c]];
        const float bl[3] = { n.bmin.x, n.bmin.y, n.bmin.z }, bh[3] = { n.bmax.x, n.bmax.y, n.bmax.z };
        for (int a = 0; a < 3; ++a) { lo[a] = hmin(lo[a], bl[a]); hi[a] = hmax(hi[a], bh[a]); }
    }
    for (int a = 0; a < 3; ++a) {
        if (!(lo[a] <= hi[a]) || !isfinite(lo[a]) || !isfinite(hi[a])) { atomicOr(error, SB_ERR_BOUNDS); return; }
        wn.base[a] = lo[a];
        int e = 1;
        if (hi[a] > lo[a]) e = min(max(extent_exponent(hi[a], lo[a]) + 127, 1), 254);
        for (;; ++e) {
            if (e > 230) { atomicOr(error, SB_ERR_RANGE); return; }
            bool ok = true;
            for (int c = 0; c < 8 && ok; ++c) {
                if (c >= nc) { wn.qlo[a][c] = 255; wn.qhi[a][c] = 0; continue; }
                const RefNode& n = nodes[T.slot_bin[c]];
                const float bl = a == 0 ? n.bmin.x : (a == 1 ? n.bmin.y : n.bmin.z);
                const float bh = a == 0 ? n.bmax.x : (a == 1 ? n.bmax.y : n.bmax.z);
                const int ql = quant_floor_x(lo[a], e - 127, bl), qh = quant_ceil_x(lo[a], e - 127, bh);
                if (qh > 255) { ok = false; break; }
                wn.qlo[a][c] = (uint8_t)ql;
                wn.qhi[a][c] = (uint8_t)qh;
            }
            if (ok) { wn.exp[a] = (uint8_t)e; break; }
        }
    }
    for (uint32_t oct = 0; oct < 8; ++oct) wn.order[oct] = visit_word(T, oct);
    const U4* src = reinterpret_cast<const U4*>(&wn);
    U4* dst = reinterpret_cast<U4*>(wide + w);
    for (int k = 0; k < WIDE_NODE_WORDS; ++k) dst[k] = src[k];
}

// Most deferred child references along any path below wide node w (build_wide_bvh's reverse sweep), one level at a time
__global__ void need_kernel(const WideNode* __restrict__ wide, uint32_t first, uint32_t n, uint32_t* __restrict__ need) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WideNode& wn = wide[first + i];
    uint32_t below = 0;
    for (int c = 0; c < wn.n_children; ++c)
        if (wn.meta[c] & META_INTERIOR) below = max(below, need[wn.child_base + (wn.meta[c] & 0x7f)]);
    need[first + i] = (wn.n_children ? wn.n_children - 1u : 0u) + below;
}

inline unsigned grid256(uint64_t n) { return (unsigned)((n + 255u) / 256u); }

// Stream-ordered device scratch, released on every path out.
struct Scratch {
    cudaStream_t s;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t st) : s(st) {}
    ~Scratch() { for (void* p : ptrs) cudaFreeAsync(p, s); }
    template <typename T> cudaError_t get(T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cudaMallocAsync(&p, std::max<size_t>(count * sizeof(T), 16), s);
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = static_cast<T*>(p);
        return e;
    }
};

// Phase times on stderr (B2RT_TRACE_BUILD): CUDA events around every phase of the build.
struct PhaseClock {
    bool on;
    cudaStream_t s;
    std::vector<cudaEvent_t> ev;
    std::vector<const char*> names;
    PhaseClock(cudaStream_t st) : on(getenv("B2RT_TRACE_BUILD") != nullptr), s(st) { mark(nullptr); }
    void mark(const char* name) {
        if (!on) return;
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) { cudaGetLastError(); on = false; return; }
        cudaEventRecord(e, s);
        ev.push_back(e);
        names.push_back(name);
    }
    void report(uint64_t n_tris) {
        if (!on || ev.size() < 2) return;
        cudaEventSynchronize(ev.back());
        fprintf(stderr, "[b2rt_build_scene_device] %llu triangles:", (unsigned long long)n_tris);
        for (size_t i = 1; i < ev.size(); ++i) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            fprintf(stderr, " %s %.3f ms%s", names[i], ms, i + 1 < ev.size() ? "," : "\n");
        }
    }
    ~PhaseClock() { for (cudaEvent_t e : ev) cudaEventDestroy(e); }
};

// Derives the compressed wide BVH of (nodes, tris) on ctx's device and moves it into ctx's derived arrays (install_scene
// follows once the new buffers are bound). Nothing of the previous scene is touched before the derivation has succeeded.
int derive_wide_device(b2rt_context* ctx, const RefNode* nodes, uint32_t n_nodes, const RefTriangle* tris, uint32_t n_tris, PhaseClock& clock,
                       DerivedScene& d) {
    cudaStream_t s = ctx->stream;
    Scratch S(s);
    int* parent; unsigned* arrivals; float* dist; uint8_t *split, *open_root;
    uint2 *items[2];
    uint32_t *cnt[3], *excl[3], *sums[3], *need, *child_bin, *leaf_dir;
    unsigned* stats;                                  // [0] error, [1] deepest binary node
    WideNode* wide;
    U4* leaf;
    // upper bounds: a wide node is rooted at a distinct binary node; a leaf block holds 3 words per triangle + 2 for a box
    const uint64_t leaf_cap = 3ull * n_tris + 2ull * n_nodes + 4;
    const uint32_t sw = (uint32_t)scan_scratch_words(n_nodes);
    CK(S.get(&parent, n_nodes)); CK(S.get(&arrivals, n_nodes)); CK(S.get(&dist, 8ull * n_nodes)); CK(S.get(&split, 8ull * n_nodes));
    CK(S.get(&open_root, n_nodes)); CK(S.get(&items[0], n_nodes)); CK(S.get(&items[1], n_nodes));
    for (int k = 0; k < 3; ++k) { CK(S.get(&cnt[k], n_nodes)); CK(S.get(&excl[k], n_nodes)); CK(S.get(&sums[k], sw)); }
    CK(S.get(&need, n_nodes)); CK(S.get(&child_bin, 8ull * n_nodes)); CK(S.get(&leaf_dir, 2ull * n_nodes)); CK(S.get(&stats, 4));
    CK(S.get(&wide, n_nodes)); CK(S.get(&leaf, leaf_cap));
    CK(cudaMemsetAsync(stats, 0, 16, s));
    plan_init_kernel<<<grid256(n_nodes), 256, 0, s>>>(nodes, n_nodes, parent, arrivals, dist, split, open_root);
    plan_up_kernel<<<grid256(n_nodes), 256, 0, s>>>(nodes, n_nodes, parent, arrivals, dist, split, open_root);
    ctx->launches += 2;
    const uint2 root_item = make_uint2(0u, 0u);
    CK(cudaMemcpyAsync(items[0], &root_item, sizeof(root_item), cudaMemcpyHostToDevice, s));
    clock.mark("cut plan");

    // levels of the host's FIFO queue: wide nodes [first, first + size), children numbered behind them in slot order
    std::vector<std::pair<uint32_t, uint32_t>> levels;
    uint32_t first = 0, size = 1, n_alloc = 1, cur = 0;
    uint64_t leaf_total = 0, blocks_total = 0;
    uint32_t host_stats[2] = { 0, 0 };
    while (size) {
        level_count_kernel<<<grid256(size), 256, 0, s>>>(items[cur], size, nodes, tris, split, open_root, cnt[0], cnt[1], cnt[2]);
        ctx->launches += 1;
        uint32_t tot[3];
        for (int k = 0; k < 3; ++k) {
            CK(scan_exclusive(cnt[k], size, excl[k], sums[k], &ctx->launches, s));
            CK(cudaMemcpyAsync(&tot[k], sums[k], 4, cudaMemcpyDeviceToHost, s));
        }
        CK(cudaMemcpyAsync(host_stats, stats, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));                             // one synchronisation per level: the next level's size
        if (host_stats[0]) break;
        if (leaf_total + tot[1] >= 0x7fffff00ull) return fail(ctx, B2RT_INVALID_ARG_VALUE, "invalid BVH: leaf buffer exceeds 31-bit word offsets");
        const LevelBases lb = { first, n_alloc, (uint32_t)leaf_total, (uint32_t)blocks_total };
        level_emit_kernel<<<grid256(size), 256, 0, s>>>(items[cur], size, lb, nodes, tris, split, open_root, excl[0], excl[1], excl[2], wide, leaf,
                                                        leaf_dir, child_bin, items[cur ^ 1], stats + 1, stats);
        ctx->launches += 1;
        CK(cudaGetLastError());
        levels.emplace_back(first, size);
        first += size;
        n_alloc += tot[0];
        leaf_total += tot[1];
        blocks_total += tot[2];
        size = tot[0];
        cur ^= 1;
    }
    CK(cudaMemcpyAsync(host_stats, stats, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (host_stats[0] & SB_ERR_BOUNDS) return fail(ctx, B2RT_INVALID_ARG_VALUE, "invalid BVH: non-finite or inverted bounds");
    if (host_stats[0] & SB_ERR_RANGE) return fail(ctx, B2RT_INVALID_ARG_VALUE, "invalid BVH: bounds too large to quantise");
    const uint32_t n_wide = n_alloc;
    for (size_t l = levels.size(); l-- > 0;)
        need_kernel<<<grid256(levels[l].second), 256, 0, s>>>(wide, levels[l].first, levels[l].second, need);
    ctx->launches += levels.size();
    uint32_t stack_entries = 0;
    CK(cudaMemcpyAsync(&stack_entries, need, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    clock.mark("wide BVH");
    const uint32_t bound = stack_entries + 1u;              // wide_stack_bound
    if (bound > 256) return fail(ctx, B2RT_OUT_OF_RESOURCES, "BVH too deep for the traversal stack (wide depth " + std::to_string(levels.size() - 1) + ")");

    // install: the same allocations as the host derivation (ensure_scene), filled on the device
    leaf_total += 4;                                         // 64 readable zero bytes behind the last block (coop.cuh)
    const size_t wb = (size_t)n_wide * sizeof(WideNode), lb = (size_t)leaf_total * sizeof(U4), sb = (size_t)n_tris * sizeof(ShadeTri);
    free_scene(ctx);
    ctx->scene_dirty = true;                                 // until install_scene: a failure from here on leaves the bound scene to be re-derived
    int st = alloc_bvh(ctx, wb, lb);
    if (st) return st;
    CK(cudaMalloc(&ctx->d_shade, std::max<size_t>(sb, 48)));
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_child_bin), std::max<size_t>((size_t)n_wide * 32, 32)));
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_leaf_dir), std::max<size_t>((size_t)blocks_total * 8, 8)));
    CK(cudaMemcpyAsync(ctx->d_wide, wide, wb, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(ctx->d_leaf, leaf, lb - 64, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemsetAsync(static_cast<char*>(ctx->d_leaf) + lb - 64, 0, 128, s));    // the trailing words and alloc_bvh's slack
    CK(cudaMemcpyAsync(ctx->d_child_bin, child_bin, (size_t)n_wide * 32, cudaMemcpyDeviceToDevice, s));
    CK(cudaMemcpyAsync(ctx->d_leaf_dir, leaf_dir, (size_t)blocks_total * 8, cudaMemcpyDeviceToDevice, s));
    CK(launch_shade_records(static_cast<ShadeTri*>(ctx->d_shade), tris, n_tris, s));
    ctx->launches += 1;
    CK(cudaStreamSynchronize(s));
    clock.mark("install");
    d.n_tris = n_tris; d.n_nodes = n_nodes; d.n_wide_nodes = n_wide; d.n_leaf_blocks = blocks_total;
    d.wide_bytes = wb; d.leaf_bytes = lb; d.shade_bytes = sb;
    d.max_depth_binary = host_stats[1]; d.max_depth_wide = (uint32_t)levels.size() - 1u; d.stack_bound = bound;
    return B2RT_SUCCESS;
}

int new_scene_buffer(b2rt_context* ctx, size_t bytes, b2rt_buffer* id) {
    if (ctx->group) return group_buffer_create(ctx, B2RT_MEM_READ_ONLY, bytes, nullptr, id);
    return buffer_create_single(ctx, B2RT_MEM_READ_ONLY, bytes, nullptr, id, false);
}

int build_scene(b2rt_context* ctx, const RefTriangle* in, uint32_t n, uint32_t* d_order_out, b2rt_buffer bufs[2], DerivedScene& d) {
    cudaStream_t s = ctx->stream;
    PhaseClock clock(s);
    Scratch S(s);
    uint32_t *flag, *group, *sums, *first, *order;
    unsigned* small;                                   // [0] error, [1..6] centroid box (ordered), [7] group count
    float* gb;
    const uint32_t sw = (uint32_t)scan_scratch_words(n);
    CK(S.get(&flag, n)); CK(S.get(&group, n)); CK(S.get(&sums, sw)); CK(S.get(&small, 8)); CK(S.get(&order, n));
    const unsigned init[8] = { 0u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u, 0u };
    CK(cudaMemcpyAsync(small, init, sizeof(init), cudaMemcpyHostToDevice, s));
    group_flag_kernel<<<grid256(n), 256, 0, s>>>(in, n, flag, small + 1, small);
    run_cap_kernel<<<grid256(n), 256, 0, s>>>(flag, n);
    CK(scan_exclusive(flag, n, group, sums, &ctx->launches, s));
    CK(cudaMemcpyAsync(small + 7, sums, 4, cudaMemcpyDeviceToDevice, s));
    unsigned host_small[8];
    CK(cudaMemcpyAsync(host_small, small, sizeof(host_small), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    ctx->launches += 2;
    if (host_small[0] & SB_ERR_VERTEX) return fail(ctx, B2RT_INVALID_ARG_VALUE, "invalid BVH: non-finite vertex positions");
    const uint32_t m = host_small[7];
    float clo[3], chi[3];
    for (int k = 0; k < 3; ++k) {
        const unsigned a = host_small[1 + k], b = host_small[4 + k];
        const unsigned ua = (a & 0x80000000u) ? (a & 0x7fffffffu) : ~a, ub = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
        memcpy(&clo[k], &ua, 4);
        memcpy(&chi[k], &ub, 4);
    }
    CK(S.get(&first, (size_t)m + 1)); CK(S.get(&gb, 6ull * m));
    scatter_first_kernel<<<grid256(n), 256, 0, s>>>(flag, group, n, sums, first);
    group_box_kernel<<<grid256(m), 256, 0, s>>>(in, first, m, gb);
    ctx->launches += 2;
    clock.mark("grouping");

    const uint64_t n_nodes = 2ull * m - 1;
    int st = new_scene_buffer(ctx, (size_t)n * sizeof(RefTriangle), &bufs[0]);
    if (st) return st;
    st = new_scene_buffer(ctx, (size_t)n_nodes * sizeof(RefNode), &bufs[1]);
    if (st) return st;
    RefTriangle* tris = static_cast<RefTriangle*>(find(ctx, bufs[0])->d_ptr);
    RefNode* nodes = static_cast<RefNode*>(find(ctx, bufs[1])->d_ptr);
    if (m == 1) {                                      // one group: the root is a leaf over every triangle (b2rt_build_bvh)
        float b[6];
        CK(cudaMemcpyAsync(b, gb, 24, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        RefNode nd;
        memset(&nd, 0, sizeof(nd));
        nd.bmin.x = b[0]; nd.bmin.y = b[1]; nd.bmin.z = b[2]; nd.bmax.x = b[3]; nd.bmax.y = b[4]; nd.bmax.z = b[5];
        nd.offset = 0;
        nd.nPrimitives = (uint16_t)n;
        std::vector<uint32_t> iota(n);
        for (uint32_t i = 0; i < n; ++i) iota[i] = i;
        CK(cudaMemcpyAsync(nodes, &nd, sizeof(nd), cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(order, iota.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));
    } else {
        void* scratch = nullptr;
        CK(S.get(reinterpret_cast<char**>(&scratch), lbvh_scratch_bytes(m)));
        CK(lbvh_build(gb, first, m, clo, chi, scratch, nodes, order, &ctx->launches, s));
    }
    clock.mark("binary BVH");
    gather_kernel<<<(unsigned)((16ull * n + 255u) / 256u), 256, 0, s>>>(reinterpret_cast<const uint4*>(in), order, n, reinterpret_cast<uint4*>(tris));
    ctx->launches += 1;
    CK(cudaGetLastError());
    if (d_order_out) CK(cudaMemcpyAsync(d_order_out, order, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
    clock.mark("re-order");
    st = derive_wide_device(ctx, nodes, (uint32_t)n_nodes, tris, n, clock, d);
    if (st) return st;
    clock.report(n);
    return B2RT_SUCCESS;
}

}  // namespace

extern "C" int b2rt_build_scene_device(b2rt_context* ctx, const void* d_triangles, uint64_t n_triangles, uint32_t* d_order_out,
                                       b2rt_buffer* triangles_out, b2rt_buffer* nodes_out, uint64_t* n_nodes_out, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!d_triangles || !n_triangles || !triangles_out || !nodes_out || !n_nodes_out) return fail(ctx, B2RT_INVALID_VALUE, "null or empty argument");
    if (n_triangles >= 0x7fffffffull) return fail(ctx, B2RT_INVALID_VALUE, "scene too large for 32-bit indices");
    // the kernels read the records with 16-byte loads: a misaligned view (e.g. a byte tensor at an odd offset) would fault
    if (reinterpret_cast<uintptr_t>(d_triangles) % 16) return fail(ctx, B2RT_INVALID_VALUE, "triangles: device address is not 16-byte aligned");
    int st = use_device(ctx);
    if (st) return st;
    cudaPointerAttributes attr;
    cudaError_t e = cudaPointerGetAttributes(&attr, d_triangles);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(ctx, B2RT_INVALID_VALUE, "triangles: not a CUDA pointer"); }
    if ((attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) || attr.device != ctx->device)
        return fail(ctx, B2RT_INVALID_VALUE, "triangles: not device memory of device " + std::to_string(ctx->device));
    if (cuda_stream && static_cast<cudaStream_t>(cuda_stream) != ctx->stream) {       // behind the caller's work on its stream
        cudaEvent_t ev = nullptr;
        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        e = cudaEventRecord(ev, static_cast<cudaStream_t>(cuda_stream));
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ev, 0);
        cudaEventDestroy(ev);
        if (e != cudaSuccess) return cuda_fail(ctx, e, "ordering behind the caller's stream");
    }
    *triangles_out = *nodes_out = 0;
    *n_nodes_out = 0;
    b2rt_buffer bufs[2] = { 0, 0 };
    const b2rt_buffer old[2] = { ctx->bound[B2RT_ARG_BUFFER_SCENE], ctx->bound[B2RT_ARG_BUFFER_NODE] };
    DerivedScene d;
    st = build_scene(ctx, static_cast<const RefTriangle*>(d_triangles), (uint32_t)n_triangles, d_order_out, bufs, d);
    // the peers of a device group get copies of the two new arrays; then slots 1 and 2 name them on every device
    if (!st && ctx->group) st = group_broadcast_buffer(ctx, bufs[0]);
    if (!st && ctx->group) st = group_broadcast_buffer(ctx, bufs[1]);
    for (int k = 0; k < 2 && !st; ++k) st = b2rt_set_arg(ctx, B2RT_ARG_BUFFER_SCENE + k, &bufs[k], sizeof(b2rt_buffer));
    if (!st) st = install_scene(ctx, d);
    if (st) {
        // the previous scene stays usable: its buffers are bound again (on every device of a group) and, as its derived
        // arrays may be gone, it is re-derived on its next use; the new buffers are released
        const std::string err = ctx->error;
        for (int k = 0; k < 2; ++k)
            if (old[k] && ctx->bound[B2RT_ARG_BUFFER_SCENE + k] != old[k] && find(ctx, old[k]))
                b2rt_set_arg(ctx, B2RT_ARG_BUFFER_SCENE + k, &old[k], sizeof(b2rt_buffer));
        for (b2rt_buffer b : bufs) if (b) b2rt_buffer_release(ctx, b);     // unbinds them where they are still bound
        ctx->scene_dirty = true;
        ctx->error = err;
        return st;
    }
    *triangles_out = bufs[0];
    *nodes_out = bufs[1];
    *n_nodes_out = d.n_nodes;
    return B2RT_SUCCESS;
}
