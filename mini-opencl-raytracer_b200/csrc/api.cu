// api.cu -- the C ABI of include/b2rt.h: context, buffers, kernel-argument slots,
// frame and ray-stream entry points. Replaces what the reference does through
// CLContext / CLKernel (CLutils.cpp:9-77). There is no CPU path in this file: a
// missing CUDA device makes b2rt_create fail and nothing else is reachable.
#include <cuda_runtime.h>
#include <atomic>
#include <thread>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <chrono>
#include <map>
#include <memory>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>
#include "b2rt.h"
#include "kernels.h"
#include "lbvh.h"
#include "wide_bvh.h"

using namespace b2rt;

#include <mutex>
#include <set>
#include "context.h"

using namespace b2rt_detail;

namespace b2rt_detail {

std::string g_create_error;

// Live handles: a buffer wrapper that outlives its context (host/runtime.cpp CLBuffer::State) must get an error from
// b2rt_buffer_release, not a use-after-free.
static std::mutex g_live_mutex;
static std::set<const b2rt_context*> g_live;
bool context_alive(const b2rt_context* ctx) { std::lock_guard<std::mutex> lk(g_live_mutex); return g_live.count(ctx) != 0; }

int fail(b2rt_context* c, int status, const std::string& msg) {
    if (c) c->error = msg; else g_create_error = msg;
    return status;
}
int cuda_fail(b2rt_context* c, cudaError_t e, const char* what) {
    int status = (e == cudaErrorMemoryAllocation) ? B2RT_MEM_OBJECT_ALLOCATION_FAILURE : B2RT_OUT_OF_RESOURCES;
    return fail(c, status, std::string(what) + ": " + cudaGetErrorString(e));
}
int use_device(b2rt_context* ctx) {
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaSetDevice");
    return B2RT_SUCCESS;
}

Buffer* find(b2rt_context* ctx, b2rt_buffer id) {
    auto it = ctx->buffers.find(id);
    return it == ctx->buffers.end() ? nullptr : &it->second;
}

void free_tail(b2rt_context* ctx) {
    for (void*& p : ctx->d_tail) { if (p) cudaFree(p); p = nullptr; }
    for (int i = 0; i < TAIL_RING + 4; ++i) ctx->tail_two_step[i] = false;
    for (int i = 0; i < TAIL_RING; ++i) { ctx->tail_slot_stream[i] = 0; ctx->tail_slot_used[i] = 0; }
}

void free_scene(b2rt_context* ctx) {
    // the tree's lines must not keep their place in the persisting part of L2 once nobody traverses it (scene_l2_setup)
    if (ctx->d_wide && ctx->l2_persist_max && ctx->opt_l2_persist) { cudaCtxResetPersistingL2Cache(); cudaGetLastError(); }
    if (ctx->d_wide) cudaFree(ctx->d_wide);          // one allocation: wide nodes, then the leaf blocks (alloc_bvh)
    if (ctx->d_shade) cudaFree(ctx->d_shade);
    if (ctx->d_child_bin) cudaFree(ctx->d_child_bin);
    if (ctx->d_leaf_dir) cudaFree(ctx->d_leaf_dir);
    ctx->d_wide = ctx->d_leaf = ctx->d_shade = nullptr;
    ctx->d_child_bin = ctx->d_leaf_dir = nullptr;
}

// Wide nodes and leaf blocks share ONE allocation (nodes first, leaf blocks behind them at a 256-byte boundary): a stream's
// L2 access-policy window is a single address range, and on scenes whose whole traversal set fits the persisting carve-out
// the window covers both (apply_l2_policy).
int alloc_bvh(b2rt_context* ctx, size_t wide_bytes, size_t leaf_bytes) {
    const size_t wb = (std::max<size_t>(wide_bytes, sizeof(WideNode)) + 255) & ~(size_t)255, lb = std::max<size_t>(leaf_bytes, 16) + 64;   // +64: slack behind the last block
    CK(cudaMalloc(&ctx->d_wide, wb + lb));
    ctx->d_leaf = static_cast<char*>(ctx->d_wide) + wb;
    ctx->bvh_bytes = wb + lb;
    return B2RT_SUCCESS;
}

// Host view of a buffer's contents: the creation-time shadow if still held, else a read-back.
int host_view(b2rt_context* ctx, Buffer* b, std::vector<uint8_t>& tmp, const uint8_t** out) {
    if (!b->shadow.empty() || b->bytes == 0) { *out = b->shadow.data(); return B2RT_SUCCESS; }
    try { tmp.resize(b->bytes); } catch (const std::bad_alloc&) { return fail(ctx, B2RT_OUT_OF_HOST_MEMORY, "host read-back buffer"); }
    CK(cudaMemcpy(tmp.data(), b->d_ptr, b->bytes, cudaMemcpyDeviceToHost));
    *out = tmp.data();
    return B2RT_SUCCESS;
}

// Build + upload the compressed wide BVH for the currently bound triangle/node buffers.
int ensure_scene(b2rt_context* ctx) {
    if (!ctx->scene_dirty) return B2RT_SUCCESS;
    Buffer* bt = find(ctx, ctx->bound[B2RT_ARG_BUFFER_SCENE]);
    Buffer* bn = find(ctx, ctx->bound[B2RT_ARG_BUFFER_NODE]);
    Buffer* bm = find(ctx, ctx->bound[B2RT_ARG_BUFFER_MATERIAL]);
    if (!bt || !bn) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "triangle (slot 1) and node (slot 2) buffers must be bound");
    if (bt->bytes % sizeof(RefTriangle) || bn->bytes % sizeof(RefNode) || bn->bytes == 0)
        return fail(ctx, B2RT_INVALID_ARG_VALUE, "scene buffers are not whole arrays of CLTriangle (256 B) / CLLinearBVHNode (48 B)");
    if (bm && bm->bytes % sizeof(RefMaterial))
        return fail(ctx, B2RT_INVALID_ARG_VALUE, "material buffer is not a whole array of CLMaterial (64 B)");
    std::vector<uint8_t> tmp_t, tmp_n;
    const uint8_t *ht = nullptr, *hn = nullptr;
    int st = host_view(ctx, bt, tmp_t, &ht);
    if (st) return st;
    st = host_view(ctx, bn, tmp_n, &hn);
    if (st) return st;
    uint64_t n_tris = bt->bytes / sizeof(RefTriangle), n_nodes = bn->bytes / sizeof(RefNode);
    WideBVH w;
    std::string err;
    try {
        err = build_wide_bvh(reinterpret_cast<const RefNode*>(hn), n_nodes, reinterpret_cast<const RefTriangle*>(ht), n_tris, w);
    } catch (const std::bad_alloc&) {
        return fail(ctx, B2RT_OUT_OF_HOST_MEMORY, "wide BVH build ran out of host memory");
    }
    if (!err.empty()) return fail(ctx, B2RT_INVALID_ARG_VALUE, "invalid BVH: " + err);
    uint32_t bound = wide_stack_bound(w);
    if (bound > 256) return fail(ctx, B2RT_OUT_OF_RESOURCES, "BVH too deep for the traversal stack (wide depth " + std::to_string(w.max_depth_wide) + ")");
    free_scene(ctx);
    size_t wb = w.nodes.size() * sizeof(WideNode), lb = w.leaf.size() * sizeof(U4), sb = w.shade.size() * sizeof(ShadeTri);
    int st_alloc = alloc_bvh(ctx, wb, lb);
    if (st_alloc) return st_alloc;
    CK(cudaMalloc(&ctx->d_shade, std::max<size_t>(sb, 48)));
    CK(cudaMemsetAsync(static_cast<char*>(ctx->d_leaf) + std::max<size_t>(lb, 16), 0, 64, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_wide, w.nodes.data(), wb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_leaf, w.leaf.data(), lb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_shade, w.shade.data(), sb, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_child_bin), std::max<size_t>(w.child_bin.size() * 4, 32)));
    CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_leaf_dir), std::max<size_t>(w.leaf_dir.size() * 4, 8)));
    CK(cudaMemcpyAsync(ctx->d_child_bin, w.child_bin.data(), w.child_bin.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_leaf_dir, w.leaf_dir.data(), w.leaf_dir.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // the 256 B/triangle host shadow is only needed for this build
    bt->shadow.clear(); bt->shadow.shrink_to_fit();
    bn->shadow.clear(); bn->shadow.shrink_to_fit();
    DerivedScene d;
    d.n_tris = n_tris; d.n_nodes = n_nodes; d.n_wide_nodes = w.nodes.size(); d.n_leaf_blocks = w.n_leaf_blocks;
    d.wide_bytes = wb; d.leaf_bytes = lb; d.shade_bytes = sb;
    d.max_depth_binary = w.max_depth_binary; d.max_depth_wide = w.max_depth_wide; d.stack_bound = bound;
    return install_scene(ctx, d);
}

int install_scene(b2rt_context* ctx, const DerivedScene& d) {
    Buffer* bt = find(ctx, ctx->bound[B2RT_ARG_BUFFER_SCENE]);
    Buffer* bn = find(ctx, ctx->bound[B2RT_ARG_BUFFER_NODE]);
    Buffer* bm = find(ctx, ctx->bound[B2RT_ARG_BUFFER_MATERIAL]);
    memset(&ctx->info, 0, sizeof(ctx->info));
    ctx->info.n_triangles = d.n_tris;
    ctx->info.n_nodes = d.n_nodes;
    ctx->info.n_materials = bm ? bm->bytes / sizeof(RefMaterial) : 0;
    ctx->info.n_wide_nodes = d.n_wide_nodes;
    ctx->info.n_leaf_blocks = d.n_leaf_blocks;
    ctx->info.wide_node_bytes = d.wide_bytes;
    ctx->info.leaf_bytes = d.leaf_bytes;
    ctx->info.shading_bytes = d.shade_bytes;
    ctx->info.max_depth_binary = d.max_depth_binary;
    ctx->info.max_depth_wide = d.max_depth_wide;
    ctx->info.sm_count = (uint32_t)ctx->sm_count;
    const uint32_t bound = d.stack_bound;
    ctx->stack_bound = bound;
    ctx->view.wide = static_cast<const U4*>(ctx->d_wide);
    ctx->view.leaf = static_cast<const U4*>(ctx->d_leaf);
    ctx->view.shade = static_cast<const ShadeTri*>(ctx->d_shade);
    ctx->view.mats = bm ? static_cast<const RefMaterial*>(bm->d_ptr) : nullptr;
    ctx->view.tris = static_cast<const RefTriangle*>(bt->d_ptr);
    ctx->view.nodes = static_cast<const RefNode*>(bn->d_ptr);
    ctx->view.n_tris = (uint32_t)d.n_tris;
    ctx->view.n_nodes = (uint32_t)d.n_nodes;
    ctx->view.n_mats = (uint32_t)ctx->info.n_materials;
    ctx->view.n_wide = (uint32_t)d.n_wide_nodes;
    ctx->view.one_bits = 0x3F800000u;
    int occ = 0;
    CK(trace_occupancy(false, bound, &occ));
    ctx->grid_closest = ctx->sm_count * std::max(occ, 1);
    CK(trace_occupancy(true, bound, &occ));
    ctx->grid_any = ctx->sm_count * std::max(occ, 1);
    scene_l2_setup(ctx);
    // cooperative tail mode: queue geometry for this tree (buffers are allocated on first use)
    free_tail(ctx);
    ctx->tail_rec_words = tail_record_words(bound);
    const int max_grid = ctx->sm_count * 32;                       // B2RT_OPT_BLOCKS_PER_SM is at most 32
    ctx->tail_capacity_records = (uint64_t)max_grid * (trace_block_threads() / 32) * COOP_MAX_LIMIT;
    CK(tail_occupancy(bound, &occ));
    ctx->grid_tail = ctx->sm_count * std::max(occ, 1);
    ctx->tuner.clear();
    ctx->tune_pending_mode = -1;
    ctx->scene_dirty = false;
    if (ctx->group) return group_adopt_scene(ctx);       // the other devices of the handle take copies over NVLink
    return B2RT_SUCCESS;
}

// The wide-node array is what every ray re-reads most (14 visits of 84 bytes per ray on the 1 M-face scene) while rays, hits
// and leaf blocks stream past it: an access-policy window marks it persisting in L2 for the kernels of `st`, so that it is
// not evicted and re-fetched from HBM (r1: 26 GB of DRAM traffic per 10^8-ray launch against 4.9 GB compulsory).
// Once per scene and device: size the persisting part of L2 to the wide-node array; the window itself is (re)applied per
// stream on first use (apply_l2_policy).
void scene_l2_setup(b2rt_context* ctx) {
    if (!ctx->l2_persist_max) return;
    // what the window covers: the whole traversal set (nodes + leaf blocks, one allocation) when it fits the persisting
    // carve-out this device allows, else the wide-node array alone (the part every ray re-reads most)
    const size_t all = ctx->bvh_bytes, nodes_only = (size_t)ctx->info.wide_node_bytes;
    ctx->l2_window_bytes = (all <= ctx->l2_persist_max && all <= ctx->l2_window_max) ? all : std::min(nodes_only, ctx->l2_window_max);
    const size_t want = (ctx->l2_window_bytes + (4u << 20)) & ~(size_t)((1u << 20) - 1);
    // (the carve-out is a property of the DEVICE: the scene set up last decides. Growing it only was tried and cost the
    // frame path of a small scene next to a large one 6-8 %: the part set aside is lost to the ray / hit queues.)
    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, ctx->opt_l2_persist ? std::min(ctx->l2_persist_max, want) : 0);
    // Lines that an EARLIER scene (of this handle or of another handle on the same device) marked persisting stay in the
    // carve-out until they are reset -- a new scene would share it with a tree nobody traverses any more.
    cudaCtxResetPersistingL2Cache();
    cudaGetLastError();
}

// Which window a stream carries is a property of the STREAM, and caller streams may be shared by several handles (bench.py
// traces two scenes on one torch stream): the table is process-wide, keyed by the stream's unique id, and a launch whose
// stream carries another scene's window (or a stale one) sets its own.
struct StreamWindow { const void* base; size_t bytes; bool persist; };
static std::mutex g_window_mutex;
static std::unordered_map<unsigned long long, StreamWindow> g_stream_windows;

int apply_l2_policy(b2rt_context* ctx, cudaStream_t st) {
    if (ctx->l2_persist_max == 0 || ctx->l2_window_max == 0 || !ctx->d_wide) return B2RT_SUCCESS;
    unsigned long long id = 0;
    if (cudaStreamGetId(st, &id) != cudaSuccess) { cudaGetLastError(); id = (unsigned long long)(uintptr_t)st; }
    id = id * 64u + (unsigned long long)(ctx->device & 63);          // stream ids are unique per process; keep devices apart anyway
    const StreamWindow want = { ctx->d_wide, ctx->l2_window_bytes, ctx->opt_l2_persist != 0 };
    {
        std::lock_guard<std::mutex> lk(g_window_mutex);
        auto it = g_stream_windows.find(id);
        // a window is an address range with properties: whoever set exactly this one, it is the right one
        if (it != g_stream_windows.end() && it->second.base == want.base && it->second.bytes == want.bytes && it->second.persist == want.persist)
            return B2RT_SUCCESS;
    }
    cudaStreamAttrValue attr;
    memset(&attr, 0, sizeof(attr));
    if (want.persist) {
        attr.accessPolicyWindow.base_ptr = ctx->d_wide;
        attr.accessPolicyWindow.num_bytes = ctx->l2_window_bytes;
        attr.accessPolicyWindow.hitRatio = std::min(1.0f, (float)ctx->l2_persist_max / (float)std::max<size_t>(attr.accessPolicyWindow.num_bytes, 1));
        attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    CK(cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr));
    {
        std::lock_guard<std::mutex> lk(g_window_mutex);
        g_stream_windows[id] = want;
        if (g_stream_windows.size() > 4096) g_stream_windows.clear();  // ids of streams long gone: start over (costs one attribute call per live stream)
    }
    return B2RT_SUCCESS;
}

// The tail queue in slot `which` (allocated on first use), wired to the given device counters. coop_max = 0 when the
// tail mode is off or the launch runs the reference-layout walk.
// Every persistent launch marks the records it writes with its own tag (never 0).
uint32_t tail_tag(b2rt_context* ctx) { if (++ctx->tail_tag_seq == 0u) ctx->tail_tag_seq = 1u; return ctx->tail_tag_seq; }

int tail_queue(b2rt_context* ctx, int which, unsigned long long* count, unsigned long long* next, TailQueue& q) {
    q = TailQueue{ count, next, nullptr, ctx->tail_rec_words, 0u, 0u, count + 2, next + 2, nullptr, count + 4, nullptr, 0u, 0u, 0u };
    // auto (-1): on; but a tree this small has no long rays -- a hand-over would cost more than the few steps it saves
    const int64_t coop = ctx->opt_coop_max >= 0 ? ctx->opt_coop_max : (ctx->info.n_wide_nodes + ctx->info.n_leaf_blocks > 1000 ? 8 : 0);
    if (coop <= 0 || ctx->opt_traversal == 1 || ctx->tail_capacity_records == 0) return B2RT_SUCCESS;
    const int64_t resume = ctx->opt_resume_max >= 0 ? ctx->opt_resume_max : 0;     // measured (r2, 10 M-face frame shares): no gain, see DESIGN.md
    const bool two_step = resume > coop;                        // a second pass only pays when it suspends earlier than the cooperative threshold
    // the queue (two of the same capacity for the two-step tail: what the first pass suspends, and what the re-packed second
    // pass leaves for the cooperative kernel) ...
    const size_t queue_words = (size_t)ctx->tail_capacity_records * ctx->tail_rec_words;
    // ... and, behind, one ticket slot per warp of the largest grid (helping warps that give a ticket back)
    const size_t orphan_slots = (size_t)ctx->tail_capacity_records / COOP_MAX_LIMIT;
    if (ctx->d_tail[which] && two_step && !ctx->tail_two_step[which]) {
        // the option was switched on after this slot was allocated with one queue: a rare, synchronous re-allocation
        CK(cudaDeviceSynchronize());
        cudaFree(ctx->d_tail[which]);
        ctx->d_tail[which] = nullptr;
    }
    if (!ctx->d_tail[which]) {
        CK(cudaMalloc(&ctx->d_tail[which], (two_step ? 2 : 1) * queue_words * sizeof(uint32_t) + orphan_slots * sizeof(unsigned long long)));
        ctx->tail_two_step[which] = two_step;
    }
    const size_t queues = ctx->tail_two_step[which] ? 2 : 1;
    q.records = static_cast<uint32_t*>(ctx->d_tail[which]);
    q.records2 = queues == 2 ? q.records + queue_words : nullptr;
    q.orphans = reinterpret_cast<unsigned long long*>(q.records + queues * queue_words);
    q.coop_max = (uint32_t)coop;
    q.resume_max = two_step ? (uint32_t)resume : 0u;
    q.tag = tail_tag(ctx);
    q.help_fcap = ctx->opt_tail_help ? 1u : 0u;                 // launch_trace_wide sizes it (or switches it off)
    return B2RT_SUCCESS;
}

// B2RT_OPT_TRAVERSAL=1: the reference-layout walk keeps one stack entry per level of the binary tree, at most 256. A tree
// that passes the wide walk's check in ensure_scene is never that deep; should one be, it is refused rather than walked
// with entries dropped.
static int binary_walk_fits(b2rt_context* ctx) {
    if (ctx->info.max_depth_binary <= 256) return B2RT_SUCCESS;
    return fail(ctx, B2RT_OUT_OF_RESOURCES, "BVH too deep for the reference-layout walk's stack (binary depth " + std::to_string(ctx->info.max_depth_binary) + ")");
}

// Grid of a persistent launch over n items: the scene's occupancy grid `base`, or B2RT_OPT_BLOCKS_PER_SM blocks per SM when
// set; `share` wavefronts running side by side each take their part of it (whole CTAs per SM); never more blocks than the
// n items fill.
static int persistent_grid(b2rt_context* ctx, int base, uint64_t n, int share = 1) {
    int grid = ctx->opt_blocks_per_sm > 0 ? ctx->sm_count * (int)ctx->opt_blocks_per_sm : base;
    if (share > 1) grid = ctx->sm_count * std::max(1, grid / ctx->sm_count / share);
    const uint64_t blocks_needed = (n + trace_block_threads() - 1) / trace_block_threads();
    return (uint64_t)grid > blocks_needed ? (int)blocks_needed : grid;
}

// B2RT_OPT_LEAF_BIAS, or the default measured for the hit policy
static uint32_t leaf_bias(const b2rt_context* ctx, bool any) { return (uint32_t)(ctx->opt_leaf_bias ? ctx->opt_leaf_bias : (any ? 48 : 32)); }

// Every launch pulls its items from its OWN counter block (a ring of NEXT_RING): launches on different caller streams may
// overlap, and a shared counter would be reset under a running kernel. Counts the launch in next_seq.
static unsigned long long* take_next(b2rt_context* ctx) { return ctx->d_next + 8 * (ctx->next_seq++ % NEXT_RING); }

// k > 0: the k nearest hits per ray (b2rt_trace_multi), d_out = b2rt_hit[n * k]; `any` is then ignored.
int trace_device(b2rt_context* ctx, const void* d_rays, uint64_t n, void* d_out, bool any, cudaStream_t st, uint32_t k = 0) {
    if (n == 0) return B2RT_SUCCESS;
    if (!d_rays || !d_out) return fail(ctx, B2RT_INVALID_VALUE, "null ray or output pointer");
    if (ctx->opt_traversal == 1) {
        int fits = binary_walk_fits(ctx);
        if (fits) return fits;
        if (k) CK(launch_trace_binary_multi(ctx->view, d_rays, n, k, d_out, ctx->info.max_depth_binary, st));
        else CK(launch_trace_binary(ctx->view, d_rays, n, d_out, any, ctx->info.max_depth_binary, st));
        ctx->launches += 1;
        return B2RT_SUCCESS;
    }
    const int grid = persistent_grid(ctx, (any && !k) ? ctx->grid_any : ctx->grid_closest, n);
    int st_pol = apply_l2_policy(ctx, st);
    if (st_pol) return st_pol;
    unsigned long long* next = take_next(ctx);
    if (k) {
        // no cooperative tail: the tail hand-over would need the row list in its record (B2RT_OPT_COOP_MAX and
        // B2RT_OPT_RESUME_MAX do not apply)
        CK(launch_trace_multi(ctx->view, d_rays, n, k, d_out, ctx->opt_counters != 0, ctx->stack_bound, grid, next, ctx->d_counters,
                              (uint32_t)ctx->opt_refill_min, leaf_bias(ctx, false), st));
        ctx->launches += 1;
        return B2RT_SUCCESS;
    }
    // Tail queues go with the STREAM: launches on one stream are ordered, so they share a queue (allocated by the first of
    // them -- r2: round robin made each of a handle's first four launches pay a 100 MB cudaMalloc, two of them inside a timed
    // region of bench.py); launches on up to TAIL_RING different streams may overlap (documented in b2rt.h), a further
    // stream takes over the queue of the stream that has not launched for longest.
    unsigned long long sid = 0;
    if (cudaStreamGetId(st, &sid) != cudaSuccess) { cudaGetLastError(); sid = (unsigned long long)(uintptr_t)st; }
    sid += 1;                                                  // 0 marks a free slot
    int slot = -1;
    for (int i = 0; i < TAIL_RING && slot < 0; ++i) if (ctx->tail_slot_stream[i] == sid) slot = i;
    if (slot < 0) {
        slot = 0;
        for (int i = 1; i < TAIL_RING; ++i) if (ctx->tail_slot_used[i] < ctx->tail_slot_used[slot]) slot = i;
        ctx->tail_slot_stream[slot] = sid;
    }
    ctx->tail_slot_used[slot] = ctx->next_seq;                 // this launch's number + 1 (take_next counted it)
    TailQueue tail;
    int st_tail = tail_queue(ctx, slot, next + 1, next + 2, tail);
    if (st_tail) return st_tail;
    CK(launch_trace_wide(ctx->view, d_rays, n, d_out, any, ctx->opt_counters != 0, ctx->stack_bound, grid, next,
                         ctx->d_counters, (uint32_t)ctx->opt_refill_min, leaf_bias(ctx, any), st, nullptr, &tail, ctx->grid_tail));
    ctx->launches += tail.coop_max ? (tail.resume_max ? 3 : 2) : 1;
    return B2RT_SUCCESS;
}

// Closest point per query (b2rt_closest_point_device): d_q = b2rt_point_query[n], d_out = b2rt_point_hit[n].
int point_device(b2rt_context* ctx, const void* d_q, uint64_t n, void* d_out, cudaStream_t st) {
    if (n == 0) return B2RT_SUCCESS;
    if (!d_q || !d_out) return fail(ctx, B2RT_INVALID_VALUE, "null query or output pointer");
    if (ctx->opt_traversal == 1) {
        int fits = binary_walk_fits(ctx);
        if (fits) return fits;
        CK(launch_closest_point_binary(ctx->view, d_q, n, d_out, ctx->info.max_depth_binary, st));
        ctx->launches += 1;
        return B2RT_SUCCESS;
    }
    const int grid = persistent_grid(ctx, ctx->grid_closest, n);
    int st_pol = apply_l2_policy(ctx, st);
    if (st_pol) return st_pol;
    unsigned long long* next = take_next(ctx);
    CK(launch_closest_point(ctx->view, d_q, n, d_out, ctx->opt_counters != 0, ctx->stack_bound, grid, next, ctx->d_counters,
                            (uint32_t)ctx->opt_refill_min, st));
    ctx->launches += 1;
    return B2RT_SUCCESS;
}

int ensure_staging(b2rt_context* ctx, uint64_t chunk, size_t out_bytes, size_t in2_bytes) {
    if (ctx->stage_capacity >= chunk && ctx->stage_out_bytes >= out_bytes && ctx->stage_in2_bytes >= in2_bytes) return B2RT_SUCCESS;
    chunk = std::max(chunk, ctx->stage_capacity);
    out_bytes = std::max(out_bytes, ctx->stage_out_bytes);
    in2_bytes = std::max(in2_bytes, ctx->stage_in2_bytes);
    for (int i = 0; i < 2; ++i) {
        if (ctx->d_stage_rays[i]) cudaFree(ctx->d_stage_rays[i]);
        if (ctx->d_stage_out[i]) cudaFree(ctx->d_stage_out[i]);
        if (ctx->d_stage_in2[i]) cudaFree(ctx->d_stage_in2[i]);
        ctx->d_stage_rays[i] = ctx->d_stage_out[i] = ctx->d_stage_in2[i] = nullptr;
    }
    ctx->stage_capacity = 0;
    ctx->stage_out_bytes = 0;
    ctx->stage_in2_bytes = 0;
    for (int i = 0; i < 2; ++i) {
        CK(cudaMalloc(&ctx->d_stage_rays[i], chunk * sizeof(b2rt_ray)));
        CK(cudaMalloc(&ctx->d_stage_out[i], out_bytes));
        if (in2_bytes) CK(cudaMalloc(&ctx->d_stage_in2[i], in2_bytes));
    }
    ctx->stage_capacity = chunk;
    ctx->stage_out_bytes = out_bytes;
    ctx->stage_in2_bytes = in2_bytes;
    return B2RT_SUCCESS;
}

// Items per pipelined chunk of the host-buffer entries; B2RT_STREAM_CHUNK (at least 1024) overrides it as a tuning aid.
static uint64_t stream_chunk() {
    if (const char* env = getenv("B2RT_STREAM_CHUNK")) { long long v = atoll(env); if (v >= 1024) return (uint64_t)v; }
    return STREAM_CHUNK;
}

// Host-buffer query stream: chunks of at most `chunk_cap` records of `in_elem` bytes (at most a b2rt_ray) are copied in,
// run through launch(d_in, d_in2, m, d_out, stream) and their `out_elem`-byte results copied out, on three streams so that
// PCIe transfers overlap the kernels. The output staging holds at least a chunk of b2rt_hit, so that every query kind fits
// the same staging buffers without reallocating. `in2` (may be NULL): a second input array of `in2_elem`-byte records,
// staged beside the first (d_in2). `what` names the input in the NULL-pointer error.
template <class Launch>
static int host_pipeline(b2rt_context* ctx, const void* in, size_t in_elem, const void* in2, size_t in2_elem, uint64_t n, void* out,
                         size_t out_elem, uint64_t chunk_cap, const char* what, Launch&& launch) {
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    if (n == 0) return B2RT_SUCCESS;
    if (!in || !out) return fail(ctx, B2RT_INVALID_VALUE, std::string("null ") + what + " or output pointer");
    const uint64_t chunk = std::min<uint64_t>(n, chunk_cap);
    st = ensure_staging(ctx, chunk, chunk * std::max(out_elem, sizeof(b2rt_hit)), in2 ? chunk * in2_elem : 0);
    if (st) return st;
    // Chunk sizes ramp up from `ramp` to `chunk` and back down at the end: the first copy-in and the last kernel +
    // copy-out are the only parts of the pipeline that nothing overlaps, so they are kept short.
    const uint64_t ramp = std::min<uint64_t>(chunk, 1ull << 19);
    uint64_t c = 0, m = 0;
    for (uint64_t off = 0; off < n; off += m, ++c) {
        const int s = (int)(c & 1);
        const uint64_t left = n - off;
        m = std::min<uint64_t>(chunk, ramp << std::min<uint64_t>(c, 16));                              // ramp up
        if (left <= ramp) m = left;
        else m = std::min<uint64_t>(m, std::max<uint64_t>(ramp, (left / 2 + 31) & ~31ull));            // ramp down: at most half of what is left
        if (c >= 2) CK(cudaStreamWaitEvent(ctx->stream_in, ctx->ev_comp[s], 0));     // in[s] free again
        CK(cudaMemcpyAsync(ctx->d_stage_rays[s], static_cast<const char*>(in) + off * in_elem, m * in_elem, cudaMemcpyHostToDevice, ctx->stream_in));
        if (in2) CK(cudaMemcpyAsync(ctx->d_stage_in2[s], static_cast<const char*>(in2) + off * in2_elem, m * in2_elem, cudaMemcpyHostToDevice, ctx->stream_in));
        CK(cudaEventRecord(ctx->ev_in[s], ctx->stream_in));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[s], 0));
        if (c >= 2) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_out[s], 0));         // out[s] drained
        st = launch(ctx->d_stage_rays[s], ctx->d_stage_in2[s], m, ctx->d_stage_out[s], ctx->stream);
        if (st) return st;
        CK(cudaEventRecord(ctx->ev_comp[s], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->stream_out, ctx->ev_comp[s], 0));
        CK(cudaMemcpyAsync(static_cast<char*>(out) + off * out_elem, ctx->d_stage_out[s], m * out_elem, cudaMemcpyDeviceToHost, ctx->stream_out));
        CK(cudaEventRecord(ctx->ev_out[s], ctx->stream_out));
    }
    CK(cudaStreamSynchronize(ctx->stream_out));
    CK(cudaStreamSynchronize(ctx->stream));
    return B2RT_SUCCESS;
}

// Host-buffer ray stream on one device. k > 0: k hits per ray (see trace_device); the chunk then shrinks with k, so that
// the output staging stays that of a closest-hit chunk.
static int trace_host(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, void* out, bool any, uint32_t k = 0) {
    uint64_t chunk = stream_chunk();
    if (k > 1) chunk = std::max<uint64_t>(chunk / k, 1024);
    const size_t out_elem = k ? (size_t)k * sizeof(b2rt_hit) : (any ? sizeof(uint32_t) : sizeof(b2rt_hit));
    return host_pipeline(ctx, rays, sizeof(b2rt_ray), nullptr, 0, n, out, out_elem, chunk, "ray",
                         [&](const void* d_in, const void*, uint64_t m, void* d_out, cudaStream_t s) { return trace_device(ctx, d_in, m, d_out, any, s, k); });
}

// Host-buffer closest-point queries on one device.
static int point_host(b2rt_context* ctx, const b2rt_point_query* q, uint64_t n, b2rt_point_hit* out) {
    return host_pipeline(ctx, q, sizeof(b2rt_point_query), nullptr, 0, n, out, sizeof(b2rt_point_hit), stream_chunk(), "query",
                         [&](const void* d_in, const void*, uint64_t m, void* d_out, cudaStream_t s) { return point_device(ctx, d_in, m, d_out, s); });
}

int frame_args(b2rt_context* ctx, FrameArgs& a);

constexpr int WF_LANES = 4;                  // concurrent wavefronts per frame launch (b2rt_context::wf_stream)
constexpr uint32_t WF_MAX_PATHS = 1u << 24;   // paths per wavefront pass (1.9 GB of queues); larger frames take several passes

void free_wavefront(b2rt_context* ctx) {
    for (int i = 0; i < 2; ++i) { if (ctx->d_wf_rays[i]) cudaFree(ctx->d_wf_rays[i]); ctx->d_wf_rays[i] = nullptr; }
    if (ctx->d_wf_hits) cudaFree(ctx->d_wf_hits);
    if (ctx->d_wf_state) cudaFree(ctx->d_wf_state);
    ctx->d_wf_hits = ctx->d_wf_state = nullptr;
    ctx->wf_capacity = 0;
}

int ensure_wavefront(b2rt_context* ctx, uint64_t paths) {
    if (!ctx->d_wf_count) CK(cudaMalloc(&ctx->d_wf_count, WF_LANES * 16 * sizeof(unsigned long long)));
    if (ctx->wf_capacity >= paths) return B2RT_SUCCESS;
    CK(cudaStreamSynchronize(ctx->stream));
    free_wavefront(ctx);
    for (int i = 0; i < 2; ++i) CK(cudaMalloc(&ctx->d_wf_rays[i], paths * sizeof(b2rt_ray)));
    CK(cudaMalloc(&ctx->d_wf_hits, paths * sizeof(b2rt_hit)));
    CK(cudaMalloc(&ctx->d_wf_state, paths * 32));
    ctx->wf_capacity = paths;
    return B2RT_SUCCESS;
}

// One wavefront over work items [0, n) of `map` on stream `s`, using the queue/state slices that start at path
// `offset` and the counter block `lane`: generate, then per bounce one persistent traversal launch over the live
// ray queue and one shade/compact launch. Queue lengths stay on the device.
// Stage timing (B2RT_OPT_STAGE_TIMES): an event after every stage of wavefront 0 of the launch; read with b2rt_stage_times.
cudaEvent_t stage_mark(b2rt_context* ctx, bool on, uint32_t kind, cudaStream_t s) {
    if (!on || ctx->stage_used >= 64) return nullptr;
    if (ctx->stage_events.size() <= ctx->stage_used) {
        cudaEvent_t ev = nullptr;
        if (cudaEventCreate(&ev) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        ctx->stage_events.push_back(ev);
        ctx->stage_kinds.push_back(0);
    }
    ctx->stage_kinds[ctx->stage_used] = kind;
    return ctx->stage_events[ctx->stage_used++];
}
#define STAGE(kind)                                                                    \
    do {                                                                               \
        if (cudaEvent_t ev__ = stage_mark(ctx, timed, (kind), s)) CK(cudaEventRecord(ev__, s)); \
    } while (0)

int wavefront_lane(b2rt_context* ctx, const FrameArgs& a, float* d_result, const GidMap& map, uint32_t n, int lane, uint64_t offset,
                   cudaStream_t s, int share, const RadianceIO* io) {
    int st_pol = apply_l2_policy(ctx, s);
    if (st_pol) return st_pol;
    const bool timed = ctx->opt_stage_times != 0 && lane == 0;
    if (timed) ctx->stage_used = 0;
    STAGE(B2RT_STAGE_BEGIN);
    unsigned long long* cnt = ctx->d_wf_count + 16 * lane;          // three rotating queue counters, the trace kernel's ray counter, its tail queues' four, the hand-over count
    char* rays[2] = { static_cast<char*>(ctx->d_wf_rays[0]) + offset * sizeof(b2rt_ray), static_cast<char*>(ctx->d_wf_rays[1]) + offset * sizeof(b2rt_ray) };
    char* hits = static_cast<char*>(ctx->d_wf_hits) + offset * sizeof(b2rt_hit);
    char* state = static_cast<char*>(ctx->d_wf_state) + offset * 32;
    CK(launch_wf_generate(a, map, n, rays[0], state, cnt, s, io));    // also resets the lane's four counters
    ctx->launches += 1;
    STAGE(B2RT_STAGE_GENERATE);
    // `share` wavefronts run side by side: each takes its part of the CTA slots (whole CTAs per SM)
    const int grid = persistent_grid(ctx, ctx->grid_closest, n, share);
    int tail_grid = ctx->grid_tail;
    if (share > 1) tail_grid = ctx->sm_count * std::max(1, tail_grid / ctx->sm_count / share);
    TailQueue tail;
    int tq = tail_queue(ctx, TAIL_RING + lane, cnt + 4, cnt + 5, tail);
    if (tq) return tq;
    for (int b = 0; b < a.bounces; ++b) {
        const int in = b & 1, out = in ^ 1;
        unsigned long long *n_in = cnt + (b % 3), *n_out = cnt + ((b + 1) % 3), *n_clear = cnt + ((b + 2) % 3);
        if (b) tail.tag = tail_tag(ctx);
        CK(launch_trace_wide(ctx->view, rays[in], n, hits, false, ctx->opt_counters != 0, ctx->stack_bound, grid,
                             cnt + 3, ctx->d_counters, (uint32_t)ctx->opt_refill_min, leaf_bias(ctx, false), s, n_in, &tail, tail_grid,
                             stage_mark(ctx, timed, B2RT_STAGE_TRACE, s)));
        STAGE(B2RT_STAGE_TAIL);
        // the shade stage also clears the counter the NEXT shade stage appends to and the traversal kernels' three counters
        CK(launch_wf_shade(ctx->view, a, map, n, rays[in], hits, n_in, rays[out], n_out, state, d_result, b == a.bounces - 1, n_clear, cnt + 3, s, io));
        ctx->launches += tail.coop_max ? (tail.resume_max ? 4 : 3) : 2;
        STAGE(B2RT_STAGE_SHADE);
    }
    return B2RT_SUCCESS;
}
#undef STAGE

// KernelEntry for work items [0, n) of `map` as up to WF_LANES independent wavefronts on their own streams. A
// stage's persistent traversal kernel ends with a tail (a few rays need 10-100x the average number of steps, on
// one lane of one warp); with several wavefronts in flight the next one's CTAs fill the SMs the tail leaves idle.
// io != null: the paths of a caller's ray stream instead of pixels (b2rt_trace_radiance, kernels.h RadianceIO).
int render_wavefront(b2rt_context* ctx, const FrameArgs& a, float* d_result, const GidMap& map, uint32_t n, const RadianceIO* io) {
    int st = ensure_wavefront(ctx, n);
    if (st) return st;
    if (a.bounces <= 0) {
        // Render() never enters its loop: radiance 0 for every pixel, which is what the megakernel does without tracing.
        CK(launch_render_mega(ctx->view, a, d_result, map, n, false, ctx->stack_bound, ctx->info.max_depth_binary, ctx->stream, io));
        ctx->launches += 1;
        return B2RT_SUCCESS;
    }
    int lanes = ctx->opt_wf_lanes > 0 ? (int)ctx->opt_wf_lanes : (n >= (1u << 20) ? 2 : 1);
    // cut at band boundaries so that every part is a GidMap again (a contiguous map can be cut anywhere)
    const bool contiguous = map.band == map.stride;
    const uint64_t unit = contiguous ? 32 : map.band;
    // ceil(n / lanes) rounded up to whole units: per * lanes >= n, so no work item is left over
    uint64_t per = (((uint64_t)n + lanes - 1) / lanes + unit - 1) / unit * unit;
    if (per == 0) per = unit;
    lanes = (int)std::min<uint64_t>(lanes, ((uint64_t)n + per - 1) / per);
    if (lanes <= 1) return wavefront_lane(ctx, a, d_result, map, n, 0, 0, ctx->stream, 1, io);
    CK(cudaEventRecord(ctx->ev_wf_fork, ctx->stream));
    for (int l = 0; l < lanes; ++l) {
        const uint64_t off = per * l, m = std::min<uint64_t>(per, n - off);
        GidMap sub = map;
        if (contiguous) { sub.begin = map.begin + off; sub.band = sub.stride = (uint32_t)m; }
        else sub.begin = map.begin + (off / map.band) * map.stride;
        CK(cudaStreamWaitEvent(ctx->wf_stream[l], ctx->ev_wf_fork, 0));
        st = wavefront_lane(ctx, a, d_result, sub, (uint32_t)m, l, off, ctx->wf_stream[l], ctx->opt_wf_grid_split ? lanes : 1, io);
        if (st) return st;
        CK(cudaEventRecord(ctx->ev_wf_join[l], ctx->wf_stream[l]));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_wf_join[l], 0));
    }
    return B2RT_SUCCESS;
}

int render_with_mode(b2rt_context* ctx, const FrameArgs& a, float* result, const GidMap& map, uint64_t n, int mode,
                     const RadianceIO* io = nullptr);
int render_tuned(b2rt_context* ctx, const FrameArgs& a, float* result, const GidMap& map, uint64_t n);

// Folds a finished timing into the tuner table. Never waits: while the timed launch is still running `*busy` is set and the
// caller simply runs another (untimed) frame in the same mode -- the host thread of an asynchronous frame loop is not
// stalled by the measurement (r1: a cudaEventSynchronize here made the first four frames of every new launch shape blocking).
int tuner_resolve(b2rt_context* ctx, bool* busy) {
    *busy = false;
    if (ctx->tune_pending_mode < 0) return B2RT_SUCCESS;
    const cudaError_t q = cudaEventQuery(ctx->ev_tune[1]);
    if (q == cudaErrorNotReady) { cudaGetLastError(); *busy = true; return B2RT_SUCCESS; }
    if (q != cudaSuccess) return cuda_fail(ctx, q, "cudaEventQuery (render-mode trial)");
    float ms = 0.0f;
    CK(cudaEventElapsedTime(&ms, ctx->ev_tune[0], ctx->ev_tune[1]));
    ModeTrial& t = ctx->tuner[ctx->tune_pending_key];
    t.ms[ctx->tune_pending_mode] = ms;
    if (ctx->tune_pending_mode == 1) t.choice = t.ms[1] < t.ms[0] ? 1 : 0;
    ctx->tune_pending_mode = -1;
    return B2RT_SUCCESS;
}

// B2RT_OPT_RENDER_MODE = 2: the wavefront and the megakernel produce bit-identical frames, so the faster one for
// THIS launch shape (work items, bounces) on THIS scene can simply be measured. Calls 1-2 of a shape run the
// wavefront, calls 3-4 the megakernel, the second of each pair between two CUDA events; once both timings have been
// read back (without waiting: cudaEventQuery at the start of a later call) the winner runs. The wavefront wins on large
// launches and incoherent scenes, the megakernel on a rank's small share of a multi-GPU frame, where the per-bounce
// stage tails of the wavefront add up.
int render_tuned(b2rt_context* ctx, const FrameArgs& a, float* result, const GidMap& map, uint64_t n) {
    bool busy = false;
    int st = tuner_resolve(ctx, &busy);
    if (st) return st;
    if (n >= WF_MAX_PATHS) return render_with_mode(ctx, a, result, map, n, 0);
    const std::pair<uint64_t, int> key(n, a.bounces);
    ModeTrial& t = ctx->tuner[key];
    if (t.choice >= 0) return render_with_mode(ctx, a, result, map, n, t.choice);
    // a trial (of this shape or another) is still in flight and owns the two events: no new measurement now
    if (busy) return render_with_mode(ctx, a, result, map, n, ctx->tune_pending_key == key ? ctx->tune_pending_mode : 0);
    const int phase = t.calls++;
    const int mode = phase < 2 ? 0 : 1;
    const bool timed = (phase & 1) != 0;
    if (timed) CK(cudaEventRecord(ctx->ev_tune[0], ctx->stream));
    st = render_with_mode(ctx, a, result, map, n, mode);
    if (st) return st;
    if (timed) {
        CK(cudaEventRecord(ctx->ev_tune[1], ctx->stream));
        ctx->tune_pending_key = key;
        ctx->tune_pending_mode = mode;
    }
    return B2RT_SUCCESS;
}

// Validates and draws the work items of `map` (n of them) into the bound output buffer.
int render_items(b2rt_context* ctx, const GidMap& map, uint64_t n) {
    int st = use_device(ctx);
    if (st) return st;
    FrameArgs a;
    st = frame_args(ctx, a);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    Buffer* out = find(ctx, ctx->bound[B2RT_ARG_BUFFER_OUT]);
    if (!out) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "output buffer (slot 0) is not bound");
    if (!ctx->view.mats || ctx->view.n_mats == 0) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "material buffer (slot 3) is not bound");
    if (n == 0) return B2RT_SUCCESS;
    if (n > 0xffffffffull || map.band == 0) return fail(ctx, B2RT_INVALID_GLOBAL_WORK_SIZE, "work size out of range");
    const uint64_t last = map.gid((uint32_t)(n - 1));
    if (last > 0xfffffffeull || (last + 1) * 16 > out->bytes)
        return fail(ctx, B2RT_INVALID_GLOBAL_WORK_SIZE, "work items up to gid " + std::to_string(last) + " exceed the output buffer (" +
                    std::to_string(out->bytes / 16) + " pixels)");
    float* result = static_cast<float*>(out->d_ptr);
    if (ctx->opt_traversal == 1) return render_with_mode(ctx, a, result, map, n, 1);
    if (ctx->opt_render_mode != 2) return render_with_mode(ctx, a, result, map, n, (int)ctx->opt_render_mode);
    return render_tuned(ctx, a, result, map, n);
}

// One frame launch in a given mode: 1 = megakernel, 0 = wavefront. io != null: a caller's ray stream (see render_wavefront).
int render_with_mode(b2rt_context* ctx, const FrameArgs& a, float* result, const GidMap& map, uint64_t n, int mode, const RadianceIO* io) {
    int st = B2RT_SUCCESS;
    if (mode == 1) {
        if (ctx->opt_traversal == 1) st = binary_walk_fits(ctx);
        if (!st) st = apply_l2_policy(ctx, ctx->stream);
        if (st) return st;
        CK(launch_render_mega(ctx->view, a, result, map, (uint32_t)n, ctx->opt_traversal == 1, ctx->stack_bound, ctx->info.max_depth_binary,
                              ctx->stream, io));
        ctx->launches += 1;
        return B2RT_SUCCESS;
    }
    // wavefront passes of at most WF_MAX_PATHS work items, each of them a GidMap again
    auto contiguous = [&](uint64_t first_gid, uint64_t count) -> int {
        for (uint64_t off = 0; off < count; off += WF_MAX_PATHS) {
            GidMap sub;
            const uint32_t m = (uint32_t)std::min<uint64_t>(WF_MAX_PATHS, count - off);
            sub.begin = first_gid + off; sub.band = sub.stride = m;
            int rc = render_wavefront(ctx, a, result, sub, m, io);
            if (rc) return rc;
        }
        return B2RT_SUCCESS;
    };
    if (map.band == map.stride) return contiguous(map.begin, n);
    if (map.band >= WF_MAX_PATHS) {
        for (uint64_t k = 0; k * map.band < n; ++k) {
            st = contiguous(map.begin + k * map.stride, std::min<uint64_t>(map.band, n - k * map.band));
            if (st) return st;
        }
        return B2RT_SUCCESS;
    }
    const uint64_t per_pass = WF_MAX_PATHS - WF_MAX_PATHS % map.band;      // whole bands
    for (uint64_t off = 0; off < n; off += per_pass) {
        GidMap sub = map;
        sub.begin = map.begin + (off / map.band) * map.stride;
        st = render_wavefront(ctx, a, result, sub, (uint32_t)std::min<uint64_t>(per_pass, n - off), io);
        if (st) return st;
    }
    return B2RT_SUCCESS;
}

// The camera part of FrameArgs: frames and b2rt_camera_rays_device make their primary rays from the same values.
static void camera_args(const b2rt_context* ctx, FrameArgs& a) {
    a.width = ctx->width; a.height = ctx->height; a.frame_count = ctx->frame_count;
    for (int k = 0; k < 3; ++k) { a.pos[k] = ctx->cam_pos[k]; a.front[k] = ctx->cam_front[k]; a.up[k] = ctx->cam_up[k]; }
    a.angle = tanf(0.5f * (45.0f * 3.1415f / 180.0f));   // kernel_bvh.cl:392, evaluated by the host libm like the oracle
}

// The shading part of FrameArgs (slots 8-10): frames and b2rt_trace_radiance shade paths with the same values.
static int shade_args(b2rt_context* ctx, FrameArgs& a) {
    for (int i : { B2RT_ARG_LIGHT_BOUNCES, B2RT_ARG_LIGHT_TYPE, B2RT_ARG_SKYBOX_INTENSITY })
        if (!ctx->arg_set[i]) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "kernel argument " + std::to_string(i) + " was never set");
    a.bounces = ctx->bounces; a.light_type = ctx->light_type; a.sky = ctx->sky;
    return B2RT_SUCCESS;
}

int frame_args(b2rt_context* ctx, FrameArgs& a) {
    for (int i = 0; i < B2RT_ARG_COUNT; ++i)
        if (!ctx->arg_set[i]) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "kernel argument " + std::to_string(i) + " was never set");
    camera_args(ctx, a);
    shade_args(ctx, a);                                  // cannot fail: every slot is set
    a.mirror = ctx->mirror;
    if (a.width == 0 || a.height == 0) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "WIDTH/HEIGHT must be non-zero");
    return B2RT_SUCCESS;
}

// Path-traced radiance per ray (b2rt_trace_radiance_device): the frame path's stages with the caller's rays and seeds as the
// source and one b2rt_radiance record per path as the sink, always on the wavefront (the megakernel over the reference-layout
// arrays with B2RT_OPT_TRAVERSAL = 1). The stages use the frame path's queues, counters and tail queues, which belong to the
// context's stream, so the launch runs there between two edges with the caller's stream.
int radiance_device(b2rt_context* ctx, const void* d_rays, const uint32_t* d_seeds, uint64_t n, void* d_out, cudaStream_t caller) {
    FrameArgs a;
    memset(&a, 0, sizeof(a));
    int st = shade_args(ctx, a);
    if (st) return st;
    if (!ctx->view.mats || ctx->view.n_mats == 0) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "material buffer (slot 3) is not bound");
    if (n == 0) return B2RT_SUCCESS;
    if (a.bounces < 0) a.bounces = 0;      // the contract's "bounces <= 0": no segment (the kernels' loop bound is unsigned)
    const RadianceIO io = { d_rays, d_seeds, d_out };
    const cudaStream_t s = ctx->stream;
    if (caller != s) CK(stream_edge(ctx->ev_refit[0], caller, s));           // behind the caller's work on its stream
    // pieces that a 32-bit work-item count holds (the megakernel's launch); render_with_mode checks the reference-layout
    // walk's stack in mode 1
    for (uint64_t off = 0; off < n && !st; off += 1ull << 31) {
        const uint64_t m = std::min<uint64_t>(n - off, 1ull << 31);
        GidMap map;
        map.begin = off;
        map.band = map.stride = (uint32_t)m;
        st = render_with_mode(ctx, a, nullptr, map, m, ctx->opt_traversal == 1 ? 1 : 0, &io);
    }
    // the caller's later work sees the records -- also after a failure, when stages that write d_out may be enqueued
    if (caller != s) CK(stream_edge(ctx->ev_refit[1], s, caller));
    return st;
}

// Host-buffer radiance on one device.
static int radiance_host(b2rt_context* ctx, const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out) {
    return host_pipeline(ctx, rays, sizeof(b2rt_ray), seeds, sizeof(uint32_t), n, out, sizeof(b2rt_radiance), stream_chunk(), "ray",
                         [&](const void* d_in, const void* d_seeds, uint64_t m, void* d_out, cudaStream_t s) {
                             return radiance_device(ctx, d_in, static_cast<const uint32_t*>(d_seeds), m, d_out, s);
                         });
}

}  // namespace b2rt_detail

// ---- lifetime ---------------------------------------------------------------------------
extern "C" int b2rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int b2rt_create(int device_id, b2rt_context** out) {
    if (!out) return fail(nullptr, B2RT_INVALID_VALUE, "null output handle");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(nullptr, B2RT_DEVICE_NOT_FOUND, std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                    " (libb2rt has no CPU fallback)");
    }
    if (device_id < 0 || device_id >= n) return fail(nullptr, B2RT_DEVICE_NOT_FOUND, "device id out of range");
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device_id)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
    if (prop.major != 10)
        return fail(nullptr, B2RT_DEVICE_NOT_FOUND, std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                    "; libb2rt ships sm_100a code only");
    b2rt_context* ctx = new (std::nothrow) b2rt_context();
    if (!ctx) return fail(nullptr, B2RT_OUT_OF_HOST_MEMORY, "context allocation");
    ctx->device = device_id;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_persist_max = (size_t)prop.persistingL2CacheMaxSize;
    ctx->l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
    memset(&ctx->info, 0, sizeof(ctx->info));
    memset(&ctx->view, 0, sizeof(ctx->view));
    auto bail = [&](cudaError_t err, const char* what) { int s = cuda_fail(nullptr, err, what); b2rt_destroy(ctx); return s; };
    if ((e = cudaSetDevice(device_id)) != cudaSuccess) return bail(e, "cudaSetDevice");
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&ctx->stream_in, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    if ((e = cudaStreamCreateWithFlags(&ctx->stream_out, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
        if ((e = cudaEventCreateWithFlags(&ctx->ev_comp[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
        if ((e = cudaEventCreateWithFlags(&ctx->ev_out[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    }
    for (int i = 0; i < 4; ++i) {
        if ((e = cudaStreamCreateWithFlags(&ctx->wf_stream[i], cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
        if ((e = cudaEventCreateWithFlags(&ctx->ev_wf_join[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    }
    if ((e = cudaEventCreateWithFlags(&ctx->ev_wf_fork, cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    for (int i = 0; i < 2; ++i) {
        if ((e = cudaEventCreate(&ctx->ev_tune[i])) != cudaSuccess) return bail(e, "cudaEventCreate");
        if ((e = cudaEventCreateWithFlags(&ctx->ev_refit[i], cudaEventDisableTiming)) != cudaSuccess) return bail(e, "cudaEventCreate");
    }
    {   // stream-ordered allocations (b2rt_build_bvh) stay mapped between calls up to 256 MB
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device_id) == cudaSuccess) {
            unsigned long long keep = 256ull << 20;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    if ((e = cudaMalloc(&ctx->d_next, NEXT_RING * 8 * sizeof(unsigned long long))) != cudaSuccess) return bail(e, "cudaMalloc");
    if ((e = cudaMalloc(&ctx->d_counters, 192)) != cudaSuccess) return bail(e, "cudaMalloc");
    if ((e = cudaMemset(ctx->d_counters, 0, 192)) != cudaSuccess) return bail(e, "cudaMemset");
    { std::lock_guard<std::mutex> lk(g_live_mutex); g_live.insert(ctx); }
    *out = ctx;
    return B2RT_SUCCESS;
}

extern "C" void b2rt_destroy(b2rt_context* ctx) {
    if (!ctx) return;
    {
        std::lock_guard<std::mutex> lk(g_live_mutex);
        if (!g_live.erase(ctx) && !ctx->stream) return;      // never registered and nothing created: a failed b2rt_create cleaning up twice
    }
    if (ctx->group) group_destroy(ctx);
    if (ctx->comm) comm_destroy(ctx);
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    free_scene(ctx);
    for (auto& kv : ctx->buffers) if (kv.second.d_ptr) cudaFree(kv.second.d_ptr);
    for (int i = 0; i < 2; ++i) {
        if (ctx->d_stage_rays[i]) cudaFree(ctx->d_stage_rays[i]);
        if (ctx->d_stage_out[i]) cudaFree(ctx->d_stage_out[i]);
        if (ctx->d_stage_in2[i]) cudaFree(ctx->d_stage_in2[i]);
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_comp[i]) cudaEventDestroy(ctx->ev_comp[i]);
        if (ctx->ev_out[i]) cudaEventDestroy(ctx->ev_out[i]);
    }
    if (ctx->d_next) cudaFree(ctx->d_next);
    if (ctx->d_counters) cudaFree(ctx->d_counters);
    free_wavefront(ctx);
    free_tail(ctx);
    if (ctx->d_wf_count) cudaFree(ctx->d_wf_count);
    if (ctx->d_rgba8) cudaFree(ctx->d_rgba8);
    for (int i = 0; i < 4; ++i) {
        if (ctx->wf_stream[i]) { cudaStreamSynchronize(ctx->wf_stream[i]); cudaStreamDestroy(ctx->wf_stream[i]); }
        if (ctx->ev_wf_join[i]) cudaEventDestroy(ctx->ev_wf_join[i]);
    }
    if (ctx->ev_wf_fork) cudaEventDestroy(ctx->ev_wf_fork);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_tune[i]) cudaEventDestroy(ctx->ev_tune[i]);
        if (ctx->ev_refit[i]) cudaEventDestroy(ctx->ev_refit[i]);
    }
    for (cudaEvent_t ev : ctx->stage_events) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->stream_in) cudaStreamDestroy(ctx->stream_in);
    if (ctx->stream_out) cudaStreamDestroy(ctx->stream_out);
    delete ctx;
}

extern "C" const char* b2rt_last_error(const b2rt_context* ctx) { return ctx ? ctx->error.c_str() : g_create_error.c_str(); }

extern "C" const char* b2rt_status_string(int status) {
    switch (status) {   // same names as GetClErrorString (CLutils.h:29-105) for the codes this library returns
        case B2RT_SUCCESS: return "CL_SUCCESS";
        case B2RT_DEVICE_NOT_FOUND: return "CL_DEVICE_NOT_FOUND";
        case B2RT_MEM_OBJECT_ALLOCATION_FAILURE: return "CL_MEM_OBJECT_ALLOCATION_FAILURE";
        case B2RT_OUT_OF_RESOURCES: return "CL_OUT_OF_RESOURCES";
        case B2RT_OUT_OF_HOST_MEMORY: return "CL_OUT_OF_HOST_MEMORY";
        case B2RT_INVALID_VALUE: return "CL_INVALID_VALUE";
        case B2RT_INVALID_CONTEXT: return "CL_INVALID_CONTEXT";
        case B2RT_INVALID_MEM_OBJECT: return "CL_INVALID_MEM_OBJECT";
        case B2RT_INVALID_ARG_INDEX: return "CL_INVALID_ARG_INDEX";
        case B2RT_INVALID_ARG_VALUE: return "CL_INVALID_ARG_VALUE";
        case B2RT_INVALID_ARG_SIZE: return "CL_INVALID_ARG_SIZE";
        case B2RT_INVALID_KERNEL_ARGS: return "CL_INVALID_KERNEL_ARGS";
        case B2RT_INVALID_GLOBAL_WORK_SIZE: return "CL_INVALID_GLOBAL_WORK_SIZE";
        default: return "Unknown OpenCL error";
    }
}

// ---- buffers and arguments --------------------------------------------------------------
extern "C" int b2rt_buffer_create(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) return group_buffer_create(ctx, flags, bytes, host_ptr, out);
    return buffer_create_single(ctx, flags, bytes, host_ptr, out, true);
}

int b2rt_detail::buffer_create_single(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out, bool zero_fill) {
    if (!out) return fail(ctx, B2RT_INVALID_VALUE, "null output buffer handle");
    *out = 0;
    if (bytes == 0) return fail(ctx, -61 /* CL_INVALID_BUFFER_SIZE */, "zero-sized buffer");
    bool copy = (flags & B2RT_MEM_COPY_HOST_PTR) != 0;
    if (copy != (host_ptr != nullptr)) return fail(ctx, -37 /* CL_INVALID_HOST_PTR */, "host_ptr and COPY_HOST_PTR must be given together");
    int st = use_device(ctx);
    if (st) return st;
    Buffer b;
    b.bytes = bytes;
    b.flags = flags;
    CK(cudaMalloc(&b.d_ptr, bytes));
    cudaError_t e;
    if (copy) {
        e = cudaMemcpyAsync(b.d_ptr, host_ptr, bytes, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e == cudaSuccess) {
            try { b.shadow.assign(static_cast<const uint8_t*>(host_ptr), static_cast<const uint8_t*>(host_ptr) + bytes); }
            catch (const std::bad_alloc&) { b.shadow.clear(); }   // fall back to a read-back at build time
        }
    } else {
        e = zero_fill ? cudaMemsetAsync(b.d_ptr, 0, bytes, ctx->stream) : cudaSuccess;
    }
    if (e != cudaSuccess) { cudaFree(b.d_ptr); return cuda_fail(ctx, e, "buffer initialisation"); }
    uint64_t id = ctx->next_id++;
    ctx->buffers.emplace(id, std::move(b));
    *out = id;
    return B2RT_SUCCESS;
}

static int buffer_release_one(b2rt_context* ctx, void* arg);

extern "C" int b2rt_buffer_release(b2rt_context* ctx, b2rt_buffer buf) {
    if (!ctx || !context_alive(ctx)) return B2RT_INVALID_CONTEXT;
    if (ctx->group) { int st = group_each(ctx, buffer_release_one, &buf, false); group_bind_output(ctx); return st; }
    return buffer_release_one(ctx, &buf);
}

static int buffer_release_one(b2rt_context* ctx, void* arg) {
    const b2rt_buffer buf = *static_cast<b2rt_buffer*>(arg);
    Buffer* b = find(ctx, buf);
    if (!b) return fail(ctx, B2RT_INVALID_MEM_OBJECT, "unknown buffer");
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(b->d_ptr);
    ctx->buffers.erase(buf);
    for (int i = 0; i < 4; ++i)
        if (ctx->bound[i] == buf) { ctx->bound[i] = 0; ctx->arg_set[i] = false; if (i) ctx->scene_dirty = true; }
    return B2RT_SUCCESS;
}

struct SetArg { uint32_t slot; const void* data; size_t size; };
static int set_arg_one(b2rt_context* ctx, uint32_t slot, const void* data, size_t size);
static int set_arg_each(b2rt_context* ctx, void* arg) { const SetArg* a = static_cast<const SetArg*>(arg); return set_arg_one(ctx, a->slot, a->data, a->size); }

extern "C" int b2rt_set_arg(b2rt_context* ctx, uint32_t slot, const void* data, size_t size) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) {
        SetArg a{ slot, data, size };
        int st = group_each(ctx, set_arg_each, &a, false);
        if (!st && slot == B2RT_ARG_BUFFER_OUT) group_bind_output(ctx);
        return st;
    }
    return set_arg_one(ctx, slot, data, size);
}

static int set_arg_one(b2rt_context* ctx, uint32_t slot, const void* data, size_t size) {
    if (slot >= B2RT_ARG_COUNT) return fail(ctx, B2RT_INVALID_ARG_INDEX, "argument index " + std::to_string(slot) + " out of range");
    if (!data) return fail(ctx, B2RT_INVALID_ARG_VALUE, "null argument value");
    static const size_t want[B2RT_ARG_COUNT] = { 8, 8, 8, 8, 4, 4, 4, 4, 4, 4, 4, 16, 16, 16 };
    if (size != want[slot])
        return fail(ctx, B2RT_INVALID_ARG_SIZE, "argument " + std::to_string(slot) + " expects " + std::to_string(want[slot]) + " bytes, got " + std::to_string(size));
    switch (slot) {
        case B2RT_ARG_BUFFER_OUT: case B2RT_ARG_BUFFER_SCENE: case B2RT_ARG_BUFFER_NODE: case B2RT_ARG_BUFFER_MATERIAL: {
            b2rt_buffer id;
            memcpy(&id, data, 8);
            if (!find(ctx, id)) return fail(ctx, B2RT_INVALID_MEM_OBJECT, "argument " + std::to_string(slot) + " is not a live buffer");
            if (ctx->bound[slot] != id && slot != B2RT_ARG_BUFFER_OUT) ctx->scene_dirty = true;
            ctx->bound[slot] = id;
            break;
        }
        case B2RT_ARG_WIDTH: memcpy(&ctx->width, data, 4); break;
        case B2RT_ARG_HEIGHT: memcpy(&ctx->height, data, 4); break;
        case B2RT_ARG_FRAME_COUNT: memcpy(&ctx->frame_count, data, 4); break;
        case B2RT_ARG_FRAME_SEED: memcpy(&ctx->frame_seed, data, 4); break;   // unused by the kernel (kernel_bvh.cl:424)
        case B2RT_ARG_LIGHT_BOUNCES: memcpy(&ctx->bounces, data, 4); break;
        case B2RT_ARG_LIGHT_TYPE: memcpy(&ctx->light_type, data, 4); break;
        case B2RT_ARG_SKYBOX_INTENSITY: memcpy(&ctx->sky, data, 4); break;
        case B2RT_ARG_CAMERA_POS: memcpy(ctx->cam_pos, data, 16); break;
        case B2RT_ARG_CAMERA_FRONT: memcpy(ctx->cam_front, data, 16); break;
        case B2RT_ARG_CAMERA_UP: memcpy(ctx->cam_up, data, 16); break;
    }
    ctx->arg_set[slot] = true;
    return B2RT_SUCCESS;
}

// ---- frame path -------------------------------------------------------------------------
extern "C" int b2rt_execute_range(b2rt_context* ctx, size_t gid_begin, size_t gid_end) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (gid_end < gid_begin || gid_end > 0xffffffffull)
        return fail(ctx, B2RT_INVALID_GLOBAL_WORK_SIZE, "bad work range [" + std::to_string(gid_begin) + "," + std::to_string(gid_end) + ")");
    if (ctx->group) return group_execute(ctx, gid_begin, gid_end);
    const uint64_t n = gid_end - gid_begin;
    GidMap map;
    map.begin = gid_begin;
    map.band = map.stride = (uint32_t)std::max<uint64_t>(n, 1);
    return render_items(ctx, map, n);
}

extern "C" int b2rt_execute_bands(b2rt_context* ctx, size_t gid_begin, uint32_t band_pixels, uint32_t stride_pixels, uint32_t n_bands) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (band_pixels == 0 || stride_pixels < band_pixels) return fail(ctx, B2RT_INVALID_GLOBAL_WORK_SIZE, "band must be non-empty and stride >= band");
    if (ctx->group) return fail(ctx, B2RT_INVALID_VALUE, "b2rt_execute_bands addresses one device; a device-group handle partitions b2rt_execute itself");
    GidMap map;
    map.begin = gid_begin;
    map.band = band_pixels;
    map.stride = stride_pixels;
    return render_items(ctx, map, (uint64_t)band_pixels * n_bands);
}

extern "C" int b2rt_execute(b2rt_context* ctx, size_t global_work_size) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (global_work_size == 0) return fail(ctx, B2RT_INVALID_GLOBAL_WORK_SIZE, "global work size is 0");
    return b2rt_execute_range(ctx, 0, global_work_size);
}

extern "C" int b2rt_read_buffer(b2rt_context* ctx, b2rt_buffer buf, void* dst, size_t bytes) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    Buffer* b = find(ctx, buf);
    if (!b) return fail(ctx, B2RT_INVALID_MEM_OBJECT, "unknown buffer");
    if (!dst || bytes > b->bytes) return fail(ctx, B2RT_INVALID_VALUE, "read of " + std::to_string(bytes) + " bytes from a " + std::to_string(b->bytes) + "-byte buffer");
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaMemcpyAsync(dst, b->d_ptr, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return B2RT_SUCCESS;
}

extern "C" int b2rt_finish(b2rt_context* ctx) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) return group_finish(ctx);
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaStreamSynchronize(ctx->stream));
    return B2RT_SUCCESS;
}

extern "C" int b2rt_host_register(b2rt_context* ctx, void* ptr, size_t bytes) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!ptr || !bytes) return fail(ctx, B2RT_INVALID_VALUE, "null or empty host range");
    int st = use_device(ctx);
    if (st) return st;
    cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return B2RT_SUCCESS; }
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaHostRegister");
    return B2RT_SUCCESS;
}
extern "C" int b2rt_host_unregister(b2rt_context* ctx, void* ptr) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!ptr) return fail(ctx, B2RT_INVALID_VALUE, "null host pointer");
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaStreamSynchronize(ctx->stream));
    cudaError_t e = cudaHostUnregister(ptr);
    if (e == cudaErrorHostMemoryNotRegistered) { cudaGetLastError(); return B2RT_SUCCESS; }
    if (e != cudaSuccess) return cuda_fail(ctx, e, "cudaHostUnregister");
    return B2RT_SUCCESS;
}

// ---- convenience --------------------------------------------------------------------------
extern "C" int b2rt_upload_scene(b2rt_context* ctx, const void* triangles, uint64_t n_triangles, const void* nodes,
                                 uint64_t n_nodes, const void* materials, uint64_t n_materials) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!triangles || !nodes || !materials || !n_triangles || !n_nodes || !n_materials)
        return fail(ctx, B2RT_INVALID_VALUE, "upload_scene needs non-empty triangle, node and material arrays");
    const void* src[3] = { triangles, nodes, materials };
    size_t bytes[3] = { (size_t)n_triangles * sizeof(RefTriangle), (size_t)n_nodes * sizeof(RefNode), (size_t)n_materials * sizeof(RefMaterial) };
    for (int i = 0; i < 3; ++i) {
        b2rt_buffer old = ctx->bound[1 + i], buf = 0;
        int st = b2rt_buffer_create(ctx, B2RT_MEM_READ_ONLY | B2RT_MEM_COPY_HOST_PTR, bytes[i], src[i], &buf);
        if (st) return st;
        st = b2rt_set_arg(ctx, 1 + i, &buf, sizeof(buf));
        if (st) return st;
        if (old && old != buf) b2rt_buffer_release(ctx, old), ctx->bound[1 + i] = buf, ctx->arg_set[1 + i] = true;
    }
    return ensure_scene(ctx);
}

extern "C" int b2rt_resize(b2rt_context* ctx, uint32_t width, uint32_t height) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!width || !height) return fail(ctx, B2RT_INVALID_VALUE, "zero frame size");
    int st = b2rt_set_arg(ctx, B2RT_ARG_WIDTH, &width, 4);
    if (st) return st;
    st = b2rt_set_arg(ctx, B2RT_ARG_HEIGHT, &height, 4);
    if (st) return st;
    b2rt_buffer old = ctx->bound[0], buf = 0;
    st = b2rt_buffer_create(ctx, B2RT_MEM_WRITE_ONLY, (size_t)width * height * 16, nullptr, &buf);
    if (st) return st;
    st = b2rt_set_arg(ctx, B2RT_ARG_BUFFER_OUT, &buf, sizeof(buf));
    if (st) return st;
    if (old) { b2rt_buffer_release(ctx, old); ctx->bound[0] = buf; ctx->arg_set[0] = true; }
    return B2RT_SUCCESS;
}

extern "C" int b2rt_read_pixels(b2rt_context* ctx, void* dst, size_t bytes) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!ctx->bound[0]) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "output buffer (slot 0) is not bound");
    return b2rt_read_buffer(ctx, ctx->bound[0], dst, bytes);
}

extern "C" int b2rt_read_pixels_rgba8(b2rt_context* ctx, void* dst, size_t bytes) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    Buffer* b = find(ctx, ctx->bound[0]);
    if (!b) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "output buffer (slot 0) is not bound");
    if (!dst || bytes % 4 || bytes / 4 > b->bytes / 16)
        return fail(ctx, B2RT_INVALID_VALUE, "8-bit read of " + std::to_string(bytes / 4) + " pixels from a " + std::to_string(b->bytes / 16) + "-pixel image");
    int st = use_device(ctx);
    if (st) return st;
    const uint64_t n = bytes / 4;
    if (n == 0) return B2RT_SUCCESS;
    if (ctx->rgba8_capacity < n) {
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->d_rgba8) cudaFree(ctx->d_rgba8);
        ctx->d_rgba8 = nullptr; ctx->rgba8_capacity = 0;
        CK(cudaMalloc(&ctx->d_rgba8, n * 4));
        ctx->rgba8_capacity = n;
    }
    CK(launch_tonemap_rgba8(b->d_ptr, ctx->d_rgba8, n, ctx->stream));
    ctx->launches += 1;
    CK(cudaMemcpyAsync(dst, ctx->d_rgba8, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return B2RT_SUCCESS;
}

// ---- device BVH build (SURVEY.md 8f-2) ----------------------------------------------------------
extern "C" int b2rt_build_bvh(b2rt_context* ctx, const void* triangles, uint64_t n_triangles, void* nodes_out, uint64_t nodes_capacity,
                              uint64_t* n_nodes_out, uint32_t* order_out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!triangles || !n_triangles || !nodes_out || !n_nodes_out || !order_out) return fail(ctx, B2RT_INVALID_VALUE, "null or empty argument");
    if (n_triangles >= 0x7fffffffull) return fail(ctx, B2RT_INVALID_VALUE, "scene too large for 32-bit indices");
    int st = use_device(ctx);
    if (st) return st;
    const RefTriangle* tris = static_cast<const RefTriangle*>(triangles);
    const bool trace = getenv("B2RT_TRACE_BUILD") != nullptr;        // developer aid: phase times on stderr
    auto now = []() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_start = now();
    // 1. groups: runs of consecutive triangles with bit-identical centroids (the loader's copies of one face). One streaming
    //    pass over the 256-byte triangles at host memory bandwidth, cut into fixed chunks that a team of threads scans
    //    independently (a run that straddles a chunk boundary becomes two groups: same centroid, adjacent Morton codes,
    //    still valid leaves; the cut points do not depend on the number of threads, so the result is deterministic).
    constexpr uint64_t CHUNK = 1u << 16;
    const uint64_t n_chunks = (n_triangles + CHUNK - 1) / CHUNK;
    struct Part { std::vector<uint32_t> first; std::vector<float> gb; float clo[3], chi[3]; };
    std::vector<Part> parts;
    std::vector<uint32_t> first;
    std::vector<float> gb;
    float clo[3] = { INFINITY, INFINITY, INFINITY }, chi[3] = { -INFINITY, -INFINITY, -INFINITY };
    try {
        parts.resize(n_chunks);
        auto scan_chunk = [&](uint64_t c) {
            Part& P = parts[c];
            const uint64_t lo_i = c * CHUNK, hi_i = std::min<uint64_t>(n_triangles, lo_i + CHUNK);
            P.first.reserve((hi_i - lo_i) / 2 + 2);
            P.gb.reserve(3 * (hi_i - lo_i) + 6);
            for (int k = 0; k < 3; ++k) { P.clo[k] = INFINITY; P.chi[k] = -INFINITY; }
            float prev[3] = { 0, 0, 0 };
            for (uint64_t i = lo_i; i < hi_i; ++i) {
                const RefVec &a = tris[i].v1.position, &b = tris[i].v2.position, &c3 = tris[i].v3.position;
                float lo[3] = { std::min(a.x, std::min(b.x, c3.x)), std::min(a.y, std::min(b.y, c3.y)), std::min(a.z, std::min(b.z, c3.z)) };
                float hi[3] = { std::max(a.x, std::max(b.x, c3.x)), std::max(a.y, std::max(b.y, c3.y)), std::max(a.z, std::max(b.z, c3.z)) };
                float cen[3] = { lo[0] * 0.5f + hi[0] * 0.5f, lo[1] * 0.5f + hi[1] * 0.5f, lo[2] * 0.5f + hi[2] * 0.5f };   // CLBVHnode.cpp:190-193
                const bool fresh = P.first.empty() || memcmp(cen, prev, 12) != 0 || i - P.first.back() >= 255;
                if (fresh) {
                    P.first.push_back((uint32_t)i);
                    P.gb.insert(P.gb.end(), { lo[0], lo[1], lo[2], hi[0], hi[1], hi[2] });
                    memcpy(prev, cen, 12);
                    for (int k = 0; k < 3; ++k) { P.clo[k] = std::min(P.clo[k], cen[k]); P.chi[k] = std::max(P.chi[k], cen[k]); }
                } else {
                    float* g = &P.gb[P.gb.size() - 6];
                    for (int k = 0; k < 3; ++k) { g[k] = std::min(g[k], lo[k]); g[3 + k] = std::max(g[3 + k], hi[k]); }
                }
            }
        };
        const unsigned team = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>({ (uint64_t)std::thread::hardware_concurrency(), n_chunks, 16 }));
        if (team <= 1) { for (uint64_t c = 0; c < n_chunks; ++c) scan_chunk(c); }
        else {
            std::atomic<uint64_t> next_chunk{ 0 };
            std::atomic<bool> oom{ false };
            std::vector<std::thread> pool;
            for (unsigned w = 0; w < team; ++w)
                pool.emplace_back([&]() {
                    try { for (uint64_t c; (c = next_chunk.fetch_add(1)) < n_chunks;) scan_chunk(c); }
                    catch (const std::bad_alloc&) { oom = true; }
                });
            for (auto& t : pool) t.join();
            if (oom) throw std::bad_alloc();
        }
        size_t total_groups = 0;
        for (const Part& P : parts) total_groups += P.first.size();
        first.reserve(total_groups + 1);
        gb.reserve(6 * total_groups);
        for (const Part& P : parts) {
            first.insert(first.end(), P.first.begin(), P.first.end());
            gb.insert(gb.end(), P.gb.begin(), P.gb.end());
            for (int k = 0; k < 3; ++k) { clo[k] = std::min(clo[k], P.clo[k]); chi[k] = std::max(chi[k], P.chi[k]); }
        }
        first.push_back((uint32_t)n_triangles);
        parts.clear();
    } catch (const std::bad_alloc&) {
        return fail(ctx, B2RT_OUT_OF_HOST_MEMORY, "BVH build ran out of host memory");
    }
    const uint32_t m = (uint32_t)first.size() - 1;
    if (nodes_capacity < 2ull * m - 1) return fail(ctx, B2RT_INVALID_VALUE, "node buffer too small: " + std::to_string(2ull * m - 1) + " nodes needed");
    RefNode* out = static_cast<RefNode*>(nodes_out);
    if (m == 1) {
        RefNode& nd = out[0];
        memset(&nd, 0, sizeof(nd));
        nd.bmin.x = gb[0]; nd.bmin.y = gb[1]; nd.bmin.z = gb[2]; nd.bmax.x = gb[3]; nd.bmax.y = gb[4]; nd.bmax.z = gb[5];
        nd.offset = 0;
        nd.nPrimitives = (uint16_t)n_triangles;
        for (uint64_t i = 0; i < n_triangles; ++i) order_out[i] = (uint32_t)i;
        *n_nodes_out = 1;
        return B2RT_SUCCESS;
    }
    const double t_grouped = now();
    // 2. Morton order, hierarchy, boxes AND the reference's flattened format on the device (lbvh.cu): 24 bytes + one index per
    //    group go up, the CLLinearBVHNode array and the triangle order come back.
    // one stream-ordered allocation for everything (the pool keeps it mapped between builds)
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    const uint64_t n_nodes = 2ull * m - 1;
    const size_t o_gb = 0, o_first = o_gb + up((size_t)m * 24), o_nodes = o_first + up((size_t)(m + 1) * 4), o_order = o_nodes + up(n_nodes * sizeof(RefNode)),
                 o_scratch = o_order + up((size_t)n_triangles * 4), total = o_scratch + up(lbvh_scratch_bytes(m));
    char* d_all = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&d_all), total, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "device BVH build allocation");
    if ((e = cudaMemcpyAsync(d_all + o_gb, gb.data(), (size_t)m * 24, cudaMemcpyHostToDevice, ctx->stream)) == cudaSuccess &&
        (e = cudaMemcpyAsync(d_all + o_first, first.data(), (size_t)(m + 1) * 4, cudaMemcpyHostToDevice, ctx->stream)) == cudaSuccess &&
        (e = lbvh_build(reinterpret_cast<const float*>(d_all + o_gb), reinterpret_cast<const uint32_t*>(d_all + o_first), m, clo, chi, d_all + o_scratch,
                        reinterpret_cast<RefNode*>(d_all + o_nodes), reinterpret_cast<uint32_t*>(d_all + o_order), &ctx->launches, ctx->stream)) == cudaSuccess &&
        (e = cudaMemcpyAsync(out, d_all + o_nodes, n_nodes * sizeof(RefNode), cudaMemcpyDeviceToHost, ctx->stream)) == cudaSuccess &&
        (e = cudaMemcpyAsync(order_out, d_all + o_order, (size_t)n_triangles * 4, cudaMemcpyDeviceToHost, ctx->stream)) == cudaSuccess)
        e = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(d_all, ctx->stream);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "device BVH build");
    if (trace) fprintf(stderr, "[b2rt_build_bvh] %llu triangles, %u groups: grouping %.1f ms, device (alloc + copies + 20 launches, flattened there) %.1f ms\n",
                       (unsigned long long)n_triangles, m, (t_grouped - t_start) * 1e3, (now() - t_grouped) * 1e3);
    *n_nodes_out = n_nodes;
    return B2RT_SUCCESS;
}

// ---- ray streams -----------------------------------------------------------------------------
// Host-buffer entries: a device group cuts the items into one contiguous range per member.
extern "C" int b2rt_trace_closest(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, b2rt_hit* hits) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) return group_split(ctx, n, [&](b2rt_context* m, uint64_t lo, uint64_t cnt) { return trace_host(m, rays + lo, cnt, hits + lo, false); });
    return trace_host(ctx, rays, n, hits, false);
}
extern "C" int b2rt_trace_any(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, uint32_t* occluded) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) return group_split(ctx, n, [&](b2rt_context* m, uint64_t lo, uint64_t cnt) { return trace_host(m, rays + lo, cnt, occluded + lo, true); });
    return trace_host(ctx, rays, n, occluded, true);
}
// Device-buffer entries: the handle's device current and its scene built; a NULL stream means the context's stream.
static int device_entry(b2rt_context* ctx, void* cuda_stream, cudaStream_t* st) {
    int s = use_device(ctx);
    if (s) return s;
    s = ensure_scene(ctx);
    if (s) return s;
    *st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream;
    return B2RT_SUCCESS;
}
extern "C" int b2rt_trace_closest_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, b2rt_hit* d_hits, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    cudaStream_t s;
    int st = device_entry(ctx, cuda_stream, &s);
    return st ? st : trace_device(ctx, d_rays, n, d_hits, false, s);
}
extern "C" int b2rt_trace_any_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, uint32_t* d_occluded, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    cudaStream_t s;
    int st = device_entry(ctx, cuda_stream, &s);
    return st ? st : trace_device(ctx, d_rays, n, d_occluded, true, s);
}
// k nearest hits: k in [1, B2RT_MULTI_MAX_HITS] and no NULL pointer with n > 0, checked before anything is touched.
static int multi_args(b2rt_context* ctx, const void* rays, uint64_t n, uint32_t k, const void* hits) {
    if (k == 0 || k > B2RT_MULTI_MAX_HITS) return fail(ctx, B2RT_INVALID_VALUE, "k must be 1.." + std::to_string(B2RT_MULTI_MAX_HITS));
    if (n && (!rays || !hits)) return fail(ctx, B2RT_INVALID_VALUE, "null ray or output pointer");
    if (n > (1ull << 56) / k) return fail(ctx, B2RT_INVALID_VALUE, "ray count too large");
    return B2RT_SUCCESS;
}
extern "C" int b2rt_trace_multi(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, uint32_t k, b2rt_hit* hits) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    int st = multi_args(ctx, rays, n, k, hits);
    if (st) return st;
    if (ctx->group) return group_split(ctx, n, [&](b2rt_context* m, uint64_t lo, uint64_t cnt) { return trace_host(m, rays + lo, cnt, hits + lo * k, false, k); });
    return trace_host(ctx, rays, n, hits, false, k);
}
extern "C" int b2rt_trace_multi_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, uint32_t k, b2rt_hit* d_hits, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    int st = multi_args(ctx, d_rays, n, k, d_hits);
    if (st) return st;
    cudaStream_t s;
    st = device_entry(ctx, cuda_stream, &s);
    return st ? st : trace_device(ctx, d_rays, n, d_hits, false, s, k);
}
// ---- closest point ----------------------------------------------------------------------------
extern "C" int b2rt_closest_point(b2rt_context* ctx, const b2rt_point_query* q, uint64_t n, b2rt_point_hit* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (n && (!q || !out)) return fail(ctx, B2RT_INVALID_VALUE, "null query or output pointer");
    if (ctx->group) return group_split(ctx, n, [&](b2rt_context* m, uint64_t lo, uint64_t cnt) { return point_host(m, q + lo, cnt, out + lo); });
    return point_host(ctx, q, n, out);
}
extern "C" int b2rt_closest_point_device(b2rt_context* ctx, const b2rt_point_query* d_q, uint64_t n, b2rt_point_hit* d_out, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (n && (!d_q || !d_out)) return fail(ctx, B2RT_INVALID_VALUE, "null query or output pointer");
    cudaStream_t s;
    int st = device_entry(ctx, cuda_stream, &s);
    return st ? st : point_device(ctx, d_q, n, d_out, s);
}
// ---- path-traced radiance ---------------------------------------------------------------------
extern "C" int b2rt_trace_radiance(b2rt_context* ctx, const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (n && (!rays || !seeds || !out)) return fail(ctx, B2RT_INVALID_VALUE, "null ray, seed or output pointer");
    if (ctx->group)
        return group_split(ctx, n, [&](b2rt_context* m, uint64_t lo, uint64_t cnt) { return radiance_host(m, rays + lo, seeds + lo, cnt, out + lo); });
    return radiance_host(ctx, rays, seeds, n, out);
}
extern "C" int b2rt_trace_radiance_device(b2rt_context* ctx, const b2rt_ray* d_rays, const uint32_t* d_seeds, uint64_t n, b2rt_radiance* d_out,
                                          void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (n && (!d_rays || !d_seeds || !d_out)) return fail(ctx, B2RT_INVALID_VALUE, "null ray, seed or output pointer");
    cudaStream_t s;
    int st = device_entry(ctx, cuda_stream, &s);
    return st ? st : radiance_device(ctx, d_rays, d_seeds, n, d_out, s);
}
extern "C" int b2rt_camera_rays_device(b2rt_context* ctx, size_t gid_begin, size_t gid_end, b2rt_ray* d_rays, void* cuda_stream) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    int st = use_device(ctx);
    if (st) return st;
    for (int i = B2RT_ARG_WIDTH; i < B2RT_ARG_COUNT; ++i) {
        if (i == B2RT_ARG_FRAME_SEED || i == B2RT_ARG_LIGHT_BOUNCES || i == B2RT_ARG_LIGHT_TYPE || i == B2RT_ARG_SKYBOX_INTENSITY) continue;
        if (!ctx->arg_set[i]) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "kernel argument " + std::to_string(i) + " was never set");
    }
    if (gid_end < gid_begin || gid_end > 0xffffffffull || !d_rays) return fail(ctx, B2RT_INVALID_VALUE, "bad camera ray range");
    FrameArgs a;
    memset(&a, 0, sizeof(a));
    camera_args(ctx, a);
    if (!a.width || !a.height) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "WIDTH/HEIGHT must be non-zero");
    CK(launch_camera_rays(a, gid_begin, gid_end, d_rays, cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream));
    ctx->launches += 1;
    return B2RT_SUCCESS;
}

// ---- introspection ------------------------------------------------------------------------------
extern "C" int b2rt_device_pointer(b2rt_context* ctx, b2rt_buffer buf, void** d_ptr, size_t* bytes) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    Buffer* b = find(ctx, buf);
    if (!b) return fail(ctx, B2RT_INVALID_MEM_OBJECT, "unknown buffer");
    if (d_ptr) *d_ptr = b->d_ptr;
    if (bytes) *bytes = b->bytes;
    return B2RT_SUCCESS;
}
extern "C" int b2rt_bound_buffer(b2rt_context* ctx, uint32_t slot, b2rt_buffer* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (slot > 3 || !out) return fail(ctx, B2RT_INVALID_ARG_INDEX, "slot is not a buffer argument");
    *out = ctx->bound[slot];
    return B2RT_SUCCESS;
}
extern "C" int b2rt_scene_info_get(b2rt_context* ctx, b2rt_scene_info* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!out) return fail(ctx, B2RT_INVALID_VALUE, "null output");
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    *out = ctx->info;
    return B2RT_SUCCESS;
}
struct SetOpt { uint32_t option; int64_t value; };
static int set_option_one(b2rt_context* ctx, uint32_t option, int64_t value);
static int set_option_each(b2rt_context* ctx, void* arg) { const SetOpt* o = static_cast<const SetOpt*>(arg); return set_option_one(ctx, o->option, o->value); }

extern "C" int b2rt_set_option(b2rt_context* ctx, uint32_t option, int64_t value) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) { SetOpt o{ option, value }; return group_each(ctx, set_option_each, &o, false); }
    return set_option_one(ctx, option, value);
}

static int set_option_one(b2rt_context* ctx, uint32_t option, int64_t value) {
    switch (option) {
        case B2RT_OPT_TRAVERSAL: if (value != 0 && value != 1) return fail(ctx, B2RT_INVALID_VALUE, "traversal must be 0 or 1"); ctx->opt_traversal = value; break;
        case B2RT_OPT_COUNTERS: ctx->opt_counters = value ? 1 : 0; break;
        case B2RT_OPT_BLOCKS_PER_SM: if (value < 0 || value > 32) return fail(ctx, B2RT_INVALID_VALUE, "blocks per SM out of range"); ctx->opt_blocks_per_sm = value; break;
        case B2RT_OPT_RENDER_MODE: if (value < 0 || value > 2) return fail(ctx, B2RT_INVALID_VALUE, "render mode must be 0 (wavefront), 1 (megakernel) or 2 (measured choice)"); ctx->opt_render_mode = value; break;
        case B2RT_OPT_WAVEFRONT_LANES: if (value < 0 || value > 4) return fail(ctx, B2RT_INVALID_VALUE, "wavefront lanes must be 0 (auto) .. 4"); ctx->opt_wf_lanes = value; break;
        case B2RT_OPT_LEAF_BIAS: if (value < 0 || value > 512) return fail(ctx, B2RT_INVALID_VALUE, "leaf bias must be 0 (default) or 1..512 (sixteenths)"); ctx->opt_leaf_bias = value; break;
        case B2RT_OPT_COOP_MAX: if (value < -1 || value > COOP_MAX_LIMIT) return fail(ctx, B2RT_INVALID_VALUE, "cooperative tail threshold must be -1 (auto), 0 (off) .. 16"); ctx->opt_coop_max = value; break;
        case B2RT_OPT_L2_PERSIST: ctx->opt_l2_persist = value ? 1 : 0; if (!ctx->scene_dirty && use_device(ctx) == B2RT_SUCCESS) { cudaStreamSynchronize(ctx->stream); scene_l2_setup(ctx); } break;
        case B2RT_OPT_RESUME_MAX: if (value < -1 || value > COOP_MAX_LIMIT) return fail(ctx, B2RT_INVALID_VALUE, "resume threshold must be -1 (auto), 0 (off) .. 16"); ctx->opt_resume_max = value; break;
        case B2RT_OPT_WAVEFRONT_GRID_SPLIT: ctx->opt_wf_grid_split = value ? 1 : 0; break;
        case B2RT_OPT_TAIL_HELP: ctx->opt_tail_help = value ? 1 : 0; break;
        case B2RT_OPT_SHARD_FENCE: ctx->opt_shard_fence = value ? 1 : 0; break;
        case B2RT_OPT_STAGE_TIMES: ctx->opt_stage_times = value ? 1 : 0; ctx->stage_used = 0; break;
        case B2RT_OPT_REFILL_MIN: if (value < 1 || value > 32) return fail(ctx, B2RT_INVALID_VALUE, "refill threshold must be 1..32"); ctx->opt_refill_min = value; break;
        default: return fail(ctx, B2RT_INVALID_VALUE, "unknown option");
    }
    ctx->tuner.clear();               // measured render-mode choices depend on the options
    ctx->tune_pending_mode = -1;
    return B2RT_SUCCESS;
}
extern "C" int b2rt_get_counters(b2rt_context* ctx, b2rt_counters* out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!out) return fail(ctx, B2RT_INVALID_VALUE, "null output");
    if (ctx->group) {                                     // sums over the devices (maxima for the per-ray maximum)
        b2rt_counters sum;
        memset(&sum, 0, sizeof(sum));
        for (b2rt_context* m : group_members(ctx)) {
            b2rt_counters c;
            Group* g = m->group;
            m->group = nullptr;
            int st = b2rt_get_counters(m, &c);
            m->group = g;
            if (st) return st;
            const uint64_t* a = reinterpret_cast<const uint64_t*>(&c);
            uint64_t* b = reinterpret_cast<uint64_t*>(&sum);
            for (size_t i = 0; i < sizeof(c) / 8; ++i) b[i] += a[i];
            sum.max_steps_per_ray = std::max(sum.max_steps_per_ray - c.max_steps_per_ray, c.max_steps_per_ray);
            sum.coop_max_steps = std::max(sum.coop_max_steps - c.coop_max_steps, c.coop_max_steps);
            sum.coop_max_rounds = std::max(sum.coop_max_rounds - c.coop_max_rounds, c.coop_max_rounds);
        }
        *out = sum;
        return B2RT_SUCCESS;
    }
    int st = use_device(ctx);
    if (st) return st;
    unsigned long long v[24];
    CK(cudaDeviceSynchronize());     // counted launches may sit on caller-provided streams
    CK(cudaMemcpy(v, ctx->d_counters, sizeof(v), cudaMemcpyDeviceToHost));
    unsigned long long ovf = 0;
    CK(stack_overflow_count(&ovf, false));
    v[13] += ovf;
    out->rays = v[0]; out->wide_nodes = v[1]; out->leaf_blocks = v[2]; out->leaf_gate_pass = v[3]; out->tri_tests = v[4];
    out->bytes_fetched = v[5] * 16ull - v[1] * 28ull;     // a node visit REQUESTS 84 of the record's 112 bytes: five 16-byte words + one of the eight order words
    out->node_phases = v[6]; out->node_phase_lanes = v[7]; out->leaf_phases = v[8]; out->leaf_phase_lanes = v[9];
    out->refills = v[10]; out->refill_lanes = v[11]; out->max_steps_per_ray = v[12];
    out->stack_overflows = v[13]; out->coop_rays = v[14]; out->coop_steps = v[15];
    out->coop_max_steps = v[16]; out->coop_max_rounds = v[17]; out->resumed_rays = v[18];
    return B2RT_SUCCESS;
}
static int reset_counters_each(b2rt_context* ctx, void*) {
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaMemsetAsync(ctx->d_counters, 0, 192, ctx->stream));
    CK(stack_overflow_count(nullptr, true));
    return B2RT_SUCCESS;
}
extern "C" int b2rt_reset_counters(b2rt_context* ctx) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group) return group_each(ctx, reset_counters_each, nullptr, false);
    int st = use_device(ctx);
    if (st) return st;
    CK(cudaMemsetAsync(ctx->d_counters, 0, 192, ctx->stream));
    return B2RT_SUCCESS;
}
extern "C" int b2rt_stage_times(b2rt_context* ctx, uint32_t* kinds, float* ms, uint32_t capacity, uint32_t* n_out) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (!kinds || !ms || !n_out) return fail(ctx, B2RT_INVALID_VALUE, "null output");
    int st = use_device(ctx);
    if (st) return st;
    *n_out = 0;
    if (ctx->stage_used < 2) return B2RT_SUCCESS;
    CK(cudaEventSynchronize(ctx->stage_events[ctx->stage_used - 1]));
    for (uint32_t i = 1; i < ctx->stage_used && *n_out < capacity; ++i) {
        float t = 0.0f;
        CK(cudaEventElapsedTime(&t, ctx->stage_events[i - 1], ctx->stage_events[i]));
        kinds[*n_out] = ctx->stage_kinds[i];
        ms[*n_out] = t;
        ++*n_out;
    }
    return B2RT_SUCCESS;
}

extern "C" uint64_t b2rt_launch_count(const b2rt_context* ctx) {
    if (!ctx) return 0;
    if (!ctx->group) return ctx->launches;
    uint64_t n = 0;
    for (const b2rt_context* m : group_members(ctx)) n += m->launches;
    return n;
}
