// kernels.cu -- hand-written sm_100a kernels behind libb2rt.so.
//
//  trace_persistent<P,COUNT,CAP>    persistent-thread while-while traversal of the
//      compressed wide BVH for a ray stream: one grid of (SMs x blocks/SM) CTAs,
//      every warp pulls chunks of rays from a global atomic counter into a
//      warp-local pool, idle lanes are re-filled from the pool with ballot/popc
//      compaction, interior-node steps and leaf steps run in separate
//      warp-uniform loops, all node/leaf fetches are 128-bit __ldg. P is the hit policy
//      (traverse.cuh): closest hit, any hit, or the k nearest hits per ray.
//  trace_binary_kernel<ANY,CAP>     one thread per ray over the reference's own
//      48 B / 256 B arrays in the reference's order: the "recompiled reference
//      kernel" baseline and an on-device cross-check of the wide path;
//      trace_binary_multi_kernel<CAP> the same walk keeping the k nearest hits.
//  camera_rays_kernel               CreateRay (kernel_bvh.cl:386-403) as a ray stream.
//  wf_generate_kernel / wf_shade_kernel   KernelEntry (kernel_bvh.cl:415-456) as a wavefront:
//      camera rays + path state, then per bounce trace_persistent over the live ray queue and
//      one shade / accumulate / compact stage; queue lengths never leave the device.
//  render_mega_kernel               KernelEntry as one launch: one thread per pixel, path loop
//      around the same traversal primitives (bit-identical to the wavefront).
//      STREAM = true (template argument of all three): the same stages with a caller's ray stream as the source and one
//      {radiance, seed} record per path as the sink (b2rt_trace_radiance).
//  tonemap_rgba8_kernel             accumulation image -> clamped 8-bit RGBA for display read-back.
//  point_persistent<COUNT,CAP>      closest point on the scene per query point (point_query.cuh), persistent like
//      trace_persistent; point_binary_kernel<CAP> the same over the reference-layout arrays, one thread per query.
//
// No tensor cores: the path is pointer chasing + fp32 slab/triangle tests, not a
// contraction (BASELINE.json north_star). Compile with -fmad=false; all
// parity-critical arithmetic additionally uses explicit *_rn intrinsics.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <type_traits>
#include "kernels.h"
#include "shade.cuh"
#include "coop.cuh"
#include "point_query.cuh"

namespace b2rt {

#ifndef B2_MIN_BLOCKS
#define B2_MIN_BLOCKS 8
#endif
static constexpr unsigned FULL = 0xffffffffu;
#ifndef B2_TOUCH
#define B2_TOUCH 0
#endif
#ifndef B2_TAIL_CODE
#define B2_TAIL_CODE 1           // 0: compile the hand-over to the cooperative tail kernel out of trace_persistent (A/B of its code-size cost)
#endif
#ifndef B2_STREAM_HINTS
#define B2_STREAM_HINTS 1
#endif
#ifndef B2_NODE_STAY_ANY
#define B2_NODE_STAY_ANY 16      // the same threshold in the any-hit kernel (r2 A/B: 16 is +2.5 % over 20 there, and -5 % for closest-hit)
#endif
#ifndef B2_NODE_STAY
#define B2_NODE_STAY 24          // (0 = off; r2 A/B: +0.9 % closest-hit at 20, +1.2 % at 24 with -0.5 % any-hit, -1.2 % at 28) > 0: consecutive node phases without a scheduling round while this many lanes want one
#endif
#ifndef B2_LEAF_STAY
#define B2_LEAF_STAY 12          // (0 = off) > 0: consecutive leaf phases without a scheduling round while this many lanes still hold a queued leaf. B200 A/B, 2^25
                                 // bench rays: closest hit +3.0 % at 12, +2.9 % at 16 and 20 over off; any-hit +5.0 / +4.7 / +3.9 %
#endif
#ifndef B2_LEAF_STAY_ANY
#define B2_LEAF_STAY_ANY 12      // the same threshold in the any-hit kernel
#endif
// "Touch" prefetch: an ordinary cached load whose result is never read, issued as soon as the next
// node / leaf of a lane is known so that the line is (on its way) in L1 when the step runs.
__device__ __forceinline__ void touch(const void* p) { unsigned d; asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(d) : "l"(p)); }
static constexpr int TRACE_BLOCK = 128;

struct RayIn { float ox, oy, oz, tmin, dx, dy, dz, tmax; };
enum { STAGE_WORDS = 11 };

__device__ __forceinline__ void load_ray(const RayIn* rays, uint64_t i, RayX& r, float& tmax) {
    // rays are read once and hits written once: streaming (evict-first) accesses keep them from displacing the
    // BVH, which every ray re-reads, from L2
    const float4* p = reinterpret_cast<const float4*>(rays + i);
#if B2_STREAM_HINTS
    float4 a = __ldcs(p), b = __ldcs(p + 1);
#else
    float4 a = __ldg(p), b = __ldg(p + 1);
#endif
    r = make_ray(a.x, a.y, a.z, b.x, b.y, b.z);
    tmax = b.w;
}

template <bool ANY>
__device__ __forceinline__ void write_result(void* __restrict__ out, uint64_t i, const HitX& h) {
#if B2_STREAM_HINTS
    if (ANY) __stcs(reinterpret_cast<uint32_t*>(out) + i, (h.tri != 0xFFFFFFFFu) ? 1u : 0u);
    else __stcs(reinterpret_cast<float4*>(out) + i, make_float4(h.t, h.u, h.v, __uint_as_float(h.tri)));
#else
    if (ANY) reinterpret_cast<uint32_t*>(out)[i] = (h.tri != 0xFFFFFFFFu) ? 1u : 0u;
    else reinterpret_cast<float4*>(out)[i] = make_float4(h.t, h.u, h.v, __uint_as_float(h.tri));
#endif
}

// A finished ray of a trace_persistent<P> launch: its hit, occlusion flag, or (HIT_MULTI) the padding of its row of k hits.
template <int P>
__device__ __forceinline__ void finish_ray(void* __restrict__ out, uint64_t i, const HitX& h, uint32_t k) {
    if (P == HIT_MULTI) pad_row(reinterpret_cast<HitX*>(out) + i * k, k, h);
    else write_result<P == HIT_ANY>(out, i, h);
}

// ---------------------------------------------------------------------------------------
// Cooperative tail (coop.cuh). trace_persistent hands the rays that are still alive when its pool is dry and a warp is
// down to a few of them to trace_tail_kernel, launched right behind it on the same stream: persistent warps pull the
// records off the queue (balanced over the whole GPU) and finish each ray with all 32 lanes.
//   record = { index lo, index hi, t, u, v, tri, n, 0, frontier[n] }   (frontier back to front, see coop_dump)
// ---------------------------------------------------------------------------------------
enum { TAIL_HEADER_WORDS = 8 };
static constexpr int TAIL_BLOCK = 128;
#ifndef B2_TAIL_MIN_BLOCKS
#define B2_TAIL_MIN_BLOCKS 8      // 64 registers: as many rays in flight as possible (the tail is latency-bound)
#endif

// What a warp serving the tail queue accumulates (the counters only in the COUNT build).
struct TailStats {
    TravCounters tc;
    unsigned long long done;
    uint32_t worst_steps, worst_rounds;
    bool overflow;
};
__device__ __forceinline__ void tail_stats_clear(TailStats& ts) {
    ts.tc = TravCounters{ 0, 0, 0, 0, 0, 0, 0 };
    ts.done = 0; ts.worst_steps = ts.worst_rounds = 0; ts.overflow = false;
}
template <bool COUNT>
__device__ __forceinline__ void tail_stats_flush(const TailStats& ts, unsigned long long* __restrict__ counters, unsigned lane) {
    if (lane != 0) return;
    if (ts.overflow) report_stack_overflow();
    if (COUNT && ts.done) {
        atomicAdd(&counters[0], ts.done);
        atomicAdd(&counters[1], (unsigned long long)ts.tc.wide_nodes); atomicAdd(&counters[2], (unsigned long long)ts.tc.leaf_blocks);
        atomicAdd(&counters[3], (unsigned long long)ts.tc.leaf_pass); atomicAdd(&counters[4], (unsigned long long)ts.tc.tri_tests);
        atomicAdd(&counters[5], (unsigned long long)ts.tc.words);
        atomicAdd(&counters[14], ts.done);                                                     // rays finished cooperatively ...
        atomicAdd(&counters[15], (unsigned long long)ts.tc.wide_nodes + ts.tc.leaf_blocks);   // ... and their node + leaf visits
        atomicMax(&counters[16], (unsigned long long)ts.worst_steps); atomicMax(&counters[17], (unsigned long long)ts.worst_rounds);
    }
}

// One record of the tail queue, finished by the whole warp. F: fcap words of this warp's shared memory. The record is read
// around L1 (ld.global.cg): a helping warp of the persistent launch reads records other SMs wrote during the same launch.
template <bool ANY, bool COUNT>
__device__ __forceinline__ void tail_process(const SceneView& s, const RayIn* __restrict__ rays, void* __restrict__ out, const uint32_t* rec,
                                             uint32_t* F, uint32_t fcap, uint32_t wide_limit, TailStats& ts) {
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t head = lane < TAIL_HEADER_WORDS ? __ldcg(rec + lane) : 0u;
    const uint64_t index = (uint64_t)__shfl_sync(FULL, head, 0) | ((uint64_t)__shfl_sync(FULL, head, 1) << 32);
    HitX h;
    h.t = __uint_as_float(__shfl_sync(FULL, head, 2)); h.u = __uint_as_float(__shfl_sync(FULL, head, 3));
    h.v = __uint_as_float(__shfl_sync(FULL, head, 4)); h.tri = __shfl_sync(FULL, head, 5);
    const uint32_t n = __shfl_sync(FULL, head, 6);
    for (uint32_t i = lane; i < n; i += 32u) F[i] = __ldcg(rec + TAIL_HEADER_WORDS + i);
    RayX r; float tmax;
    load_ray(rays, index, r, tmax);                                 // every lane: the same 32 bytes, the same arithmetic
    __syncwarp();
    const uint32_t steps0 = ts.tc.wide_nodes + ts.tc.leaf_blocks, rounds0 = ts.tc.rounds;
    coop_trace<ANY, COUNT>(s.wide, s.leaf, F, n, fcap, wide_limit, r, h, ts.tc, ts.overflow);
    if (COUNT) {
        const uint32_t ds = ts.tc.wide_nodes + ts.tc.leaf_blocks - steps0, dr = ts.tc.rounds - rounds0;
        ts.worst_steps = ts.worst_steps > ds ? ts.worst_steps : ds; ts.worst_rounds = ts.worst_rounds > dr ? ts.worst_rounds : dr;
#ifdef B2_DEBUG_LONG_RAYS
        if (dr > 300 && lane == 0) printf("LONGRAY idx %llu steps %u rounds %u o %.9g %.9g %.9g d %.9g %.9g %.9g inv %g %g %g t %g tri %u\n", (unsigned long long)index, ds, dr, r.ox, r.oy, r.oz, r.dx, r.dy, r.dz, r.ix, r.iy, r.iz, h.t, h.tri);
#endif
    }
    if (lane == 0) write_result<ANY>(out, index, h);
    ++ts.done;
    __syncwarp();
}

template <bool ANY, bool COUNT>
__global__ void __launch_bounds__(TAIL_BLOCK, B2_TAIL_MIN_BLOCKS)
trace_tail_kernel(SceneView s, const RayIn* __restrict__ rays, void* __restrict__ out, TailQueue tail,
                  unsigned long long* __restrict__ counters, uint32_t fcap, uint32_t wide_limit) {
    extern __shared__ uint32_t tail_frontiers[];                        // fcap words per warp
    uint32_t* F = tail_frontiers + (threadIdx.x >> 5) * fcap;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned long long total = *tail.count;
    TailStats ts;
    tail_stats_clear(ts);
    // tickets that helping warps of the persistent launch drew and gave back (their records were not written in time)
    if (tail.help_fcap) {
        const unsigned long long n_orphans = tail.handed[2], warps = (unsigned long long)gridDim.x * (TAIL_BLOCK / 32);
        for (unsigned long long i = (unsigned long long)blockIdx.x * (TAIL_BLOCK / 32) + (threadIdx.x >> 5); i < n_orphans; i += warps) {
            const unsigned long long slot = tail.orphans[i];
            if (slot < total) tail_process<ANY, COUNT>(s, rays, out, tail.records + slot * tail.rec_words, F, fcap, wide_limit, ts);
        }
    }
    for (;;) {
        unsigned long long slot = 0;
        if (lane == 0) slot = atomicAdd(tail.next, 1ull);
        slot = __shfl_sync(FULL, slot, 0);
        if (slot >= total) break;
        tail_process<ANY, COUNT>(s, rays, out, tail.records + slot * tail.rec_words, F, fcap, wide_limit, ts);
    }
    tail_stats_flush<COUNT>(ts, counters, lane);
}

#ifndef B2_TAIL_NOINLINE
#define B2_TAIL_NOINLINE 1      // measured (r2 A/B, 10^8-ray stream): inlined 2 840 Mrays/s, not inlined 2 885 = the kernel without any hand-over code
#endif
// The hand-over of one unfinished ray: index, best hit so far and pending work (in the reference's depth-first order) go to
// the tail queue; a whole warp finishes it (a helping warp of this launch, or trace_tail_kernel). The tag goes in last,
// behind a fence: whoever sees it sees the record.
#if B2_TAIL_NOINLINE
__device__ __noinline__
#else
__device__ __forceinline__
#endif
void tail_handover(const TailQueue& tail, uint64_t index, float t, float u, float v, uint32_t tri, uint32_t cur, uint32_t leaf0,
                   uint32_t leaf1, uint32_t top, int sp, const uint32_t* stack) {
    const unsigned long long slot = atomicAdd(tail.count, 1ull);
    uint32_t* rec = tail.records + slot * tail.rec_words;
    rec[0] = (uint32_t)index; rec[1] = (uint32_t)(index >> 32);
    rec[2] = __float_as_uint(t); rec[3] = __float_as_uint(u); rec[4] = __float_as_uint(v); rec[5] = tri;
    rec[6] = coop_dump_fields(sp, top, cur, leaf1, leaf0, stack, rec + TAIL_HEADER_WORDS);      // the frontier, back to front
    __threadfence();
    *reinterpret_cast<volatile uint32_t*>(rec + 7) = tail.tag;
}

// A suspended ray comes back: best hit so far and the frontier of the record, see Lane::resume. Not inlined (the refill
// path runs once per ray) and handed back by value: a Lane whose address escaped would live in local memory for good.
struct ResumeState { float t, u, v; uint32_t tri, cur, leaf0, leaf1, top; int sp; };
template <class LaneT>
__device__ __noinline__ ResumeState resume_fetch(uint32_t* stack, const uint32_t* __restrict__ rec) {
    static_assert(B2_LEAF_QUEUE == 2, "Lane::resume deals out a two-leaf queue");
    LaneT T;
    T.resume(stack, rec + TAIL_HEADER_WORDS, rec[6]);
    ResumeState o;
    o.t = __uint_as_float(rec[2]); o.u = __uint_as_float(rec[3]); o.v = __uint_as_float(rec[4]); o.tri = rec[5];
    o.cur = T.cur; o.leaf0 = T.leaf0; o.leaf1 = T.leaf1; o.top = T.top; o.sp = T.sp;
    return o;
}

#ifndef B2_STAGE_RAYS
#define B2_STAGE_RAYS 1          // ray set-up (InitRay: one square root, six divisions) done by all 32 lanes for the next 32 rays of the warp's pool and parked in shared memory; a refill is then eleven shared-memory loads
#endif
#ifndef B2_SMEM_STACK
#define B2_SMEM_STACK 12         // entries of every lane's traversal stack kept in shared memory (HybridStack, traverse.cuh); 0 = all in local memory
#endif
#ifndef B2_TAIL_HELP
#define B2_TAIL_HELP 0           // 1: warps that are past their hand-over serve the tail queue inside the persistent launch (epilogue of trace_persistent). Measured on a
                                 // rank's eighth of the 10 M-face 4K frame: 4.23-4.30 ms against 3.86-3.93 with the separate tail kernel -- the warps of a stage reach their hand-over
                                 // within ~0.1 ms of each other, so there is nobody free to help early, and the queue is then served less evenly than by a fresh grid. Off; kept for scenes
                                 // whose stages end less abruptly (B2RT_OPT_TAIL_HELP has an effect only in a build with 1).
#endif
#ifndef B2_HELP_POLLS
#define B2_HELP_POLLS 64         // empty polls (~0.5 us apart) a helping warp makes before it gives up: never an unbounded wait on CTAs that may not be resident
#endif
enum { WARP_SMEM_WORDS = (B2_SMEM_STACK + (B2_STAGE_RAYS ? STAGE_WORDS : 0)) * 32 };   // shared memory of one warp of trace_persistent: stack columns, then the staged rays

// ---------------------------------------------------------------------------------------
// Persistent speculative while-while traversal.
//
// Every lane owns one ray (Lane<> in traverse.cuh). Per iteration the warp votes: lanes whose
// next action is a wide-node test vs lanes holding a queued leaf. The majority action runs for
// the lanes that want it (a lane with a queued leaf AND a node to test can join either), so most
// issued instructions have many active lanes even though rays are incoherent. Finished lanes are
// re-filled from a warp-local pool of ray indices (ballot + popc compaction) that is topped up
// from one global atomic counter, `chunk` rays at a time.
// HIT_MULTI (k hits per ray, out = HitX[n * k]): each lane keeps its ray's list in the ray's own output row; such launches
// have no cooperative tail and no two-step resume (a dry warp stays until every lane is idle), k is a launch argument.
// ---------------------------------------------------------------------------------------
template <int P, bool COUNT, int CAP>
__global__ void __launch_bounds__(TRACE_BLOCK, B2_MIN_BLOCKS)
trace_persistent(SceneView s, const RayIn* __restrict__ rays, uint64_t n, void* __restrict__ out,
                 unsigned long long* __restrict__ next, unsigned long long* __restrict__ counters, uint32_t chunk,
                 uint32_t refill_min, uint32_t leaf_bias, const unsigned long long* __restrict__ n_dev, TailQueue tail,
                 const uint32_t* __restrict__ resume, uint32_t k) {
    constexpr bool ANY = P == HIT_ANY, MULTI = P == HIT_MULTI;
    // resume != null: the "rays" of this launch are the hand-over records of a previous one (n_dev = their count): every
    // lane picks a suspended ray up where its first owner left it
    const unsigned lane = threadIdx.x & 31u;
    if (n_dev) {
        // wavefront stages: the ray count is the previous stage's queue counter, never seen by the host
        n = *n_dev;
        if (n == 0) return;
        const uint64_t c = n / ((uint64_t)gridDim.x * (TRACE_BLOCK / 32) * 8u + 1u);
        chunk = (uint32_t)(c < 32 ? 32 : (c > 512 ? 512 : (c & ~31ull)));
    }
#if B2_TAIL_CODE && B2_TAIL_HELP
    if (tail.help_fcap && lane == 0) atomicAdd(tail.handed + 1, 1ull);           // "started", see the helping epilogue
#endif
    Lane<P, COUNT, CAP> L;
    uint32_t local_stack[CAP];
    // One contiguous piece of shared memory per warp: [stack entry][lane] columns, then the staged rays; the whole piece is
    // the frontier of a helping warp once its own rays are done (epilogue).
#if B2_SMEM_STACK || B2_STAGE_RAYS
    __shared__ uint32_t smem_warps[(TRACE_BLOCK / 32) * WARP_SMEM_WORDS];
    uint32_t* const smem_warp = smem_warps + (threadIdx.x >> 5) * WARP_SMEM_WORDS;
#endif
#if B2_SMEM_STACK
    const HybridStack<B2_SMEM_STACK, 32> stack = { smem_warp + lane, local_stack };
#else
    uint32_t* const stack = local_stack;
#endif
#if B2_STAGE_RAYS
    // [word][slot] per warp: o, d (normalised), 1/d, tmax, sign -- the slot of ray i is i mod 32 (the staged rays are the
    // next <= 32 of the warp's contiguous pool, so the slots are distinct)
    uint32_t* const stage = smem_warp + B2_SMEM_STACK * 32;
    // Staged at any time: the rays of the pool that share pool_next's block of 32 indices (pool chunks start at multiples of
    // 32), set up when pool_next enters the block -- no extra state.
#endif
    L.clear();
    L.overflow = false;
    L.tc.wide_nodes = L.tc.leaf_blocks = L.tc.leaf_pass = L.tc.tri_tests = L.tc.words = L.tc.max_stack = L.tc.rounds = 0;
    uint64_t my_index = 0;
    uint32_t has_out = 0;                    // this lane's finished ray still has to be written (done together with the next refill)
    uint64_t pool_next = 0;                  // warp-uniform: next ray of the warp's pool ...
    uint32_t pool_left = 0;                  // ... and how many it still holds; POOL_DRY once the global counter has run past n
    // warp-uniform: the number of idle lanes at which the warp leaves the step loop -- refill_min while the pool can still be
    // topped up, 32 - coop_max (hand-over to the cooperative tail; 32 = only when every lane is idle) once it has run dry.
    // One compare per scheduling round instead of the refill / finished / hand-over conditions one by one.
    uint32_t leave_at = refill_min;
    const uint32_t POOL_DRY = 0xffffffffu;   // pools are only topped up when empty, so "the counter ran past n" and "nothing left to hand out" coincide
    uint32_t traced = 0;
    uint32_t ray_steps = 0, max_ray_steps = 0;   // COUNT only: node + leaf steps of the current ray / the worst ray of this lane
    uint32_t ph_node = 0, ph_node_lanes = 0, ph_leaf = 0, ph_leaf_lanes = 0, ph_refill = 0, ph_refill_lanes = 0;   // COUNT only, warp-uniform

    // A lane is idle exactly when its Lane is done(): a live ray always wants a node or a leaf step.
    for (;;) {
        const unsigned vn = __ballot_sync(FULL, L.wants_node());
        const unsigned vl = __ballot_sync(FULL, L.wants_leaf());
        const unsigned busy = vn | vl;
        if (32u - (unsigned)__popc(busy) >= leave_at) {
            // nothing in flight and nothing left to fetch, or (tail) nothing left to fetch and only a few rays alive in this
            // warp: leave; those rays are handed to the cooperative tail kernel below
            if (pool_left == POOL_DRY) break;
            // ---- refill idle lanes from the warp pool -------------------------------------------
            // Finished rays are written here, several lanes at a time, instead of one lane at a time when they finish.
            const unsigned idle = ~busy;
            if (has_out) { finish_ray<P>(out, my_index, L.h, k); has_out = 0; }
            if (pool_left == 0u) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(next, (unsigned long long)chunk);
                base = __shfl_sync(FULL, base, 0);
                if (base >= n) { pool_left = POOL_DRY; leave_at = (B2_TAIL_CODE && !MULTI) ? 32u - (tail.coop_max < 31u ? tail.coop_max : 31u) : 32u; continue; }
                pool_next = base;
                pool_left = (base + chunk < n) ? chunk : (uint32_t)(n - base);
            }
#if B2_STAGE_RAYS
            if (!resume) {
                const uint32_t in_block = 32u - ((uint32_t)pool_next & 31u);
                const uint32_t staged = pool_left < in_block ? pool_left : in_block;
                if (in_block == 32u && pool_left) {
                    // set-up of the next rays of the pool on all lanes at once, busy ones included: 1/32 of InitRay per ray
                    // instead of 1/(refilled lanes), and one wait for HBM per 32 rays
                    if (lane < staged) {
                        const uint64_t i = pool_next + lane;
                        RayX r; float tmax;
                        load_ray(rays, i, r, tmax);
                        uint32_t* q = stage + ((uint32_t)i & 31u);
                        q[0 * 32] = __float_as_uint(r.ox); q[1 * 32] = __float_as_uint(r.oy); q[2 * 32] = __float_as_uint(r.oz);
                        q[3 * 32] = __float_as_uint(r.dx); q[4 * 32] = __float_as_uint(r.dy); q[5 * 32] = __float_as_uint(r.dz);
                        q[6 * 32] = __float_as_uint(r.ix); q[7 * 32] = __float_as_uint(r.iy); q[8 * 32] = __float_as_uint(r.iz);
                        q[9 * 32] = __float_as_uint(tmax); q[10 * 32] = r.sign;
                    }
                    __syncwarp();
                }
                const unsigned rank = __popc(idle & ((1u << lane) - 1u));
                if (((idle >> lane) & 1u) && rank < staged) {
                    my_index = pool_next + rank;
                    const uint32_t* q = stage + ((uint32_t)my_index & 31u);
                    RayX r;
                    r.ox = __uint_as_float(q[0 * 32]); r.oy = __uint_as_float(q[1 * 32]); r.oz = __uint_as_float(q[2 * 32]);
                    r.dx = __uint_as_float(q[3 * 32]); r.dy = __uint_as_float(q[4 * 32]); r.dz = __uint_as_float(q[5 * 32]);
                    r.ix = __uint_as_float(q[6 * 32]); r.iy = __uint_as_float(q[7 * 32]); r.iz = __uint_as_float(q[8 * 32]);
                    r.sign = q[10 * 32];
                    L.start(r, __uint_as_float(q[9 * 32]));
                }
                const unsigned taken = __popc(idle), used = (taken < staged) ? taken : staged;
                if (COUNT && used) { ph_refill++; ph_refill_lanes += used; }
                __syncwarp();                                      // the slots are read before the next staging overwrites them
                pool_next += used;
                pool_left -= used;
            } else
#endif
            {
                const uint32_t avail = pool_left;
                if (avail) {
                    const unsigned rank = __popc(idle & ((1u << lane) - 1u));
                    if (((idle >> lane) & 1u) && rank < avail) {
                        my_index = pool_next + rank;
                        const uint32_t* rec = nullptr;
                        if (resume) {
                            rec = resume + my_index * tail.rec_words;
                            my_index = (uint64_t)rec[0] | ((uint64_t)rec[1] << 32);
                        }
                        RayX r; float tmax;
                        load_ray(rays, my_index, r, tmax);
                        L.start(r, tmax);
                        if (resume) {
                            const ResumeState o = resume_fetch<Lane<P, COUNT, CAP>>(local_stack, rec);
                            L.h.t = o.t; L.h.u = o.u; L.h.v = o.v; L.h.tri = o.tri;
                            L.cur = o.cur; L.leaf0 = o.leaf0; L.leaf1 = o.leaf1; L.top = o.top; L.sp = o.sp;
#if B2_SMEM_STACK
                            for (int i = 0; i < L.sp && i < B2_SMEM_STACK; ++i) stk_set(stack, i, local_stack[i]);
#endif
                        }
                    }
                    const unsigned taken = __popc(idle), used = (taken < avail) ? taken : avail;
                    if (COUNT) { ph_refill++; ph_refill_lanes += used; if (resume && lane == 0) atomicAdd(&counters[18], (unsigned long long)used); }
                    pool_next += used;
                    pool_left -= used;
                }
            }
            continue;
        }

        // leaf_bias/16 weighs the leaf vote: > 1 consumes queued leaves earlier (less speculation)
        bool stepped;
        if (__popc(vn) * 16u >= __popc(vl) * leaf_bias) {
#if B2_NODE_STAY
            // Node phases come in runs: while at least B2_NODE_STAY lanes still want a node test, the warp goes straight
            // into the next one -- one ballot instead of the whole scheduling round (idle / refill / tail checks, leaf vote).
            unsigned want = vn;
            do {
                if (COUNT) { ph_node++; ph_node_lanes += __popc(want); }
                stepped = L.wants_node();
                if (stepped) L.node_step(s.wide, stack, s.one_bits);
                if (COUNT && stepped) ray_steps++;
                if (stepped && L.done()) {
                    has_out = 1;
                    if (COUNT) { traced++; max_ray_steps = max_ray_steps > ray_steps ? max_ray_steps : ray_steps; ray_steps = 0; }
                }
                want = __ballot_sync(FULL, L.wants_node());
            } while ((unsigned)__popc(want) >= (unsigned)(ANY ? B2_NODE_STAY_ANY : B2_NODE_STAY));
            continue;
#else
            if (COUNT) { ph_node++; ph_node_lanes += __popc(vn); }
            stepped = L.wants_node();
            if (stepped) L.node_step(s.wide, stack, s.one_bits);
#endif
        } else {
#if B2_LEAF_STAY
            // leaf phases in runs, the same way (B2_LEAF_STAY)
            unsigned want = vl;
            do {
                if (COUNT) { ph_leaf++; ph_leaf_lanes += __popc(want); }
                stepped = L.wants_leaf();
                if (stepped) L.leaf_step(s.leaf, stack, MULTI ? reinterpret_cast<HitX*>(out) + my_index * k : nullptr, k);
                if (COUNT && stepped) ray_steps++;
                if (stepped && L.done()) {
                    has_out = 1;
                    if (COUNT) { traced++; max_ray_steps = max_ray_steps > ray_steps ? max_ray_steps : ray_steps; ray_steps = 0; }
                }
                want = __ballot_sync(FULL, L.wants_leaf());
            } while ((unsigned)__popc(want) >= (unsigned)(ANY ? B2_LEAF_STAY_ANY : B2_LEAF_STAY));
            continue;
#else
            if (COUNT) { ph_leaf++; ph_leaf_lanes += __popc(vl); }
            stepped = L.wants_leaf();
            if (stepped) L.leaf_step(s.leaf, stack, MULTI ? reinterpret_cast<HitX*>(out) + my_index * k : nullptr, k);
#endif
        }
#if B2_TOUCH
        if (stepped) {
            if (L.wants_node()) { touch(s.wide + (uint32_t)WIDE_NODE_WORDS * L.cur); if (B2_TOUCH > 1) touch(s.wide + (uint32_t)WIDE_NODE_WORDS * L.cur + 6); }
            if (L.wants_leaf()) touch(s.leaf + (L.leaf0 & ~REF_LEAF_BIT));
        }
#endif
        if (COUNT && stepped) ray_steps++;
        if (stepped && L.done()) {
            has_out = 1;
            if (COUNT) { traced++; max_ray_steps = max_ray_steps > ray_steps ? max_ray_steps : ray_steps; ray_steps = 0; }
        }
    }
    if (has_out) finish_ray<P>(out, my_index, L.h, k);       // rays that finished after the last refill
    // at most coop_max lanes per warp get here, and the queue holds coop_max records per warp of the grid
    if (B2_TAIL_CODE && !MULTI && tail.coop_max && !L.done()) {
#if B2_SMEM_STACK
        for (int i = 0; i < L.sp && i < B2_SMEM_STACK; ++i) local_stack[i] = stk_get(stack, i);      // the record wants one plain array
#endif
        tail_handover(tail, my_index, L.h.t, L.h.u, L.h.v, L.h.tri, L.cur, L.leaf0, L.leaf1, L.top, L.sp, local_stack);
    }
#if B2_TAIL_CODE && B2_TAIL_HELP && (B2_SMEM_STACK || B2_STAGE_RAYS)
    // ---- helping -----------------------------------------------------------------------------------------------------------
    // This warp's rays are finished or handed over, while other warps of the launch may walk on for a long time (a stage of a
    // frame share is a few rays per lane: its end is most of it). Instead of leaving, the warp serves the tail queue: it takes
    // the records that are completely written (tag), in queue order, and finishes each with all 32 lanes -- the tail kernel's
    // work, started while the queue is still filling. It leaves when every warp of the grid is past its hand-over and the
    // queue is empty, or after B2_HELP_POLLS empty polls: no unbounded wait, so nothing depends on the whole grid being
    // resident; whatever is left in the queue is the tail kernel's, as before.
    if (!MULTI && tail.coop_max && tail.help_fcap) {
        __syncwarp();
        TailStats ts;
        tail_stats_clear(ts);
        const unsigned long long total_warps = (unsigned long long)gridDim.x * (TRACE_BLOCK / 32);
        volatile unsigned long long* const v_handed = tail.handed;            // warps past their hand-over
        volatile unsigned long long* const v_started = tail.handed + 1;       // warps that have begun (all of them: the whole grid is resident)
        volatile unsigned long long* const v_next = tail.next;
        volatile unsigned long long* const v_count = tail.count;
        if (lane == 0) { __threadfence(); atomicAdd(tail.handed, 1ull); }
        const uint32_t fcap = tail.help_fcap, wide_limit = tail.help_wide_limit;
        for (;;) {
            // Lane 0 looks (plain reads) and, if there may be a record, draws a ticket: one atomic per claim, and a ticket
            // beyond the records written so far simply waits for ITS record -- no herd of failing compare-and-swaps on one
            // word (measured: 4 700 warps retrying a CAS per record made a 0.7 ms stage take 120 ms).
            uint32_t take = 0;
            unsigned long long slot = 0;
            if (lane == 0) {
                uint32_t polls = 0;
                bool ticket = false;
                for (;;) {
                    const bool all_here = *v_started >= total_warps, all_handed = *v_handed >= total_warps;
                    if (!ticket) {
                        if (*v_next < *v_count) { slot = atomicAdd(tail.next, 1ull); ticket = true; continue; }
                        // nothing to claim: wait for more only if every producer is resident and some are still walking
                        if (all_handed || !all_here || ++polls > (uint32_t)B2_HELP_POLLS) break;
                    } else {
                        if (*reinterpret_cast<volatile uint32_t*>(tail.records + slot * tail.rec_words + 7) == tail.tag) { take = 1; break; }
                        if (all_handed && slot >= *v_count) break;            // a ticket past the final count: there is no such record
                        if (!all_here || ++polls > (uint32_t)B2_HELP_POLLS) {
                            // not waiting on CTAs that may not be resident: the ticket goes to the tail kernel's list
                            tail.orphans[atomicAdd(tail.handed + 2, 1ull)] = slot;
                            break;
                        }
                    }
                    __nanosleep(polls < 8u ? 500u : 4000u);
                }
            }
            take = __shfl_sync(FULL, take, 0);
            if (!take) break;
            slot = __shfl_sync(FULL, slot, 0);
            __threadfence();
            tail_process<ANY, COUNT>(s, rays, out, tail.records + slot * tail.rec_words, smem_warp, fcap, wide_limit, ts);
        }
        tail_stats_flush<COUNT>(ts, counters, lane);
    }
#endif

    if (COUNT) {
        if (L.overflow) report_stack_overflow();             // counting build only, see Lane::push
        // one atomic per counter per warp
        unsigned long long v[6] = { traced, L.tc.wide_nodes, L.tc.leaf_blocks, L.tc.leaf_pass, L.tc.tri_tests, L.tc.words };
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            unsigned long long x = v[i];
            for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
            if (lane == 0 && x) atomicAdd(&counters[i], x);
        }
        atomicMax(&counters[12], (unsigned long long)max_ray_steps);
        if (lane == 0) {
            const unsigned long long ph[6] = { ph_node, ph_node_lanes, ph_leaf, ph_leaf_lanes, ph_refill, ph_refill_lanes };
            for (int i = 0; i < 6; ++i) if (ph[i]) atomicAdd(&counters[6 + i], ph[i]);
        }
    }
}

// ---------------------------------------------------------------------------------------
// Reference-layout binary walk (kernel_bvh.cl:171-219 verbatim semantics), except for the stack: the reference's is
// int[64] and unchecked, so on a tree deeper than 64 levels it writes past its end. This one has CAP entries, CAP at least
// the tree's binary depth (the walk holds at most one entry per level of the current path), like the oracle's growing stack.
// P = HIT_MULTI: the k nearest hits go to `row` (h holds the list's state, traverse.cuh); the caller pads the row.
// ---------------------------------------------------------------------------------------
template <int P, int CAP>
__device__ __forceinline__ HitX trace_binary(const RefTriangle* __restrict__ tris, const RefNode* __restrict__ nodes,
                                             const RayX& r, float tmax, HitX* row = nullptr, uint32_t k = 0) {
    constexpr bool ANY = P == HIT_ANY;
    HitX h; h.t = tmax; h.u = 0.0f; h.v = 0.0f; h.tri = 0xFFFFFFFFu;
    if (P == HIT_MULTI) { h.u = tmax; h.tri = 0u; }
    uint32_t stack[CAP];
    int sp = 0;
    uint32_t cur = 0;
    for (;;) {
        const float4* np = reinterpret_cast<const float4*>(nodes + cur);
        float4 lo = __ldg(np), hi = __ldg(np + 1);
        uint4 tail = __ldg(reinterpret_cast<const uint4*>(np + 2));
        uint32_t nprim = tail.y & 0xffffu, axis = (tail.y >> 16) & 0xffu;
        bool descend = false;
        if (box_gate_exact(r, lo.x, lo.y, lo.z, hi.x, hi.y, hi.z, h.t)) {
            if (nprim > 0) {
                for (uint32_t i = 0; i < nprim; ++i) {
                    const float4* tp = reinterpret_cast<const float4*>(tris + tail.x + i);
                    float4 a = __ldg(tp), b = __ldg(tp + 5), c = __ldg(tp + 10);   // positions at +0, +80, +160 B
                    if (P == HIT_MULTI) tri_test_multi(r, a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z, tail.x + i, h, row, k);
                    else tri_test_exact(r, a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z, tail.x + i, h);
                }
                if (ANY && h.tri != 0xFFFFFFFFu) break;
            } else {
                descend = true;
                bool second_first = (r.sign >> axis) & 1u;
                if (sp < CAP) stack[sp++] = second_first ? cur + 1u : tail.x;
                else report_stack_overflow();           // never: the launch picks CAP >= the binary depth (b2rt_counters::stack_overflows)
                cur = second_first ? tail.x : cur + 1u;
            }
        }
        if (!descend) {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    return h;
}

template <bool ANY, int CAP>
__global__ void __launch_bounds__(128)
trace_binary_kernel(SceneView s, const RayIn* __restrict__ rays, uint64_t n, void* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RayX r; float tmax;
    load_ray(rays, i, r, tmax);
    HitX h = trace_binary<ANY, CAP>(s.tris, s.nodes, r, tmax);
    if (ANY) reinterpret_cast<uint32_t*>(out)[i] = (h.tri != 0xFFFFFFFFu) ? 1u : 0u;
    else reinterpret_cast<float4*>(out)[i] = make_float4(h.t, h.u, h.v, __uint_as_float(h.tri));
}

template <int CAP>
__global__ void __launch_bounds__(128)
trace_binary_multi_kernel(SceneView s, const RayIn* __restrict__ rays, uint64_t n, HitX* __restrict__ out, uint32_t k) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RayX r; float tmax;
    load_ray(rays, i, r, tmax);
    HitX* row = out + i * k;
    pad_row(row, k, trace_binary<HIT_MULTI, CAP>(s.tris, s.nodes, r, tmax, row, k));
}

// ---------------------------------------------------------------------------------------
// Camera rays and the frame megakernel.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
camera_rays_kernel(FrameArgs a, uint64_t gid0, uint64_t gid1, RayIn* __restrict__ rays) {
    uint64_t g = gid0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= gid1) return;
    uint32_t gid = (uint32_t)g;
    uint32_t seed = gid + hash_u32(a.frame_count);
    V3 d = camera_dir(a, gid, seed);
    // InitRay normalises once more (kernel_bvh.cl:402,44); emit that direction.
    RayX r = make_ray(a.pos[0], a.pos[1], a.pos[2], d.x, d.y, d.z);
    float4* p = reinterpret_cast<float4*>(rays + (g - gid0));
    p[0] = make_float4(r.ox, r.oy, r.oz, 0.0f);
    p[1] = make_float4(r.dx, r.dy, r.dz, 100000.0f);
}

// One iteration of Render()'s loop after Intersect() returned `h` for ray `r` (kernel_bvh.cl:356-382).
// Returns true when the path goes on; (next_o, next_d) are then the arguments of the reference's InitRay for
// the next ray (direction NOT yet normalised by InitRay). Shared by the megakernel and the wavefront shade
// stage so that both replay exactly the same arithmetic.
__device__ __forceinline__ bool path_step(const SceneView& s, const FrameArgs& a, const RayX& r, const HitX& h, V3& radiance,
                                          V3& beta, uint32_t& seed, V3& next_o, V3& next_d) {
    if (h.tri == 0xFFFFFFFFu) {
        float sky = xmul(0.5f, a.sky);
        radiance = vadd(radiance, vmul(beta, v3(sky, sky, sky)));
        return false;
    }
    V3 o = v3(r.ox, r.oy, r.oz), d = v3(r.dx, r.dy, r.dz);
    V3 pos = vadd(o, vscale(d, h.t));
    V3 normal = hit_normal(s.shade, h);
    uint32_t mtl = s.shade[h.tri].mtl;
    if (mtl >= s.n_mats) mtl = s.n_mats - 1u;      // the reference reads out of bounds here (usemtl miss)
    const RefMaterial m = s.mats[mtl];
    radiance = vadd(radiance, vscale(vmul(beta, ldv(m.emission)), 50.0f));
    V3 wi = v3(0.0f, 0.0f, 0.0f), wo = vneg(d);
    float pdf = 0.0f;
    V3 f = sample_brdf(wo, wi, pdf, normal, m, seed);
    if (pdf <= 0.0f || pdf != pdf) return false;
    beta = vmul(beta, vdiv(vscale(f, vdot(wi, normal)), pdf));
    float lp = light_pixel(o, d, h.t, normal, a.light_type);
    radiance = vadd(radiance, vmul(vmul(v3(lp, lp, lp), ldv(m.diffuse)), beta));
    next_o = vadd(pos, vscale(wi, 0.01f));                                // kernel_bvh.cl:380
    next_d = wi;
    return true;
}

// Where a path of the frame kernels starts and where its radiance goes. STREAM = false (frames): the camera ray of pixel
// g with seed g + hash(frame_count), segment 0 bounded by B2RT_MAX_RENDER_DIST, radiance into the running average of the
// pixel. STREAM = true (b2rt_trace_radiance): the caller's ray g with its tmax and RNG state io.seeds[g]; the record
// {radiance, seed after the path} goes to io.out[g].
__device__ __forceinline__ void stream_path_start(const RadianceIO& io, uint64_t g, float4& q0, float4& q1, uint32_t& seed) {
    const float4* p = static_cast<const float4*>(io.rays) + 2 * g;
    q0 = __ldcs(p); q1 = __ldcs(p + 1);
    seed = __ldcs(io.seeds + g);
}
__device__ __forceinline__ void store_radiance(const RadianceIO& io, uint64_t g, V3 radiance, uint32_t seed) {
    __stcs(static_cast<float4*>(io.out) + g, make_float4(radiance.x, radiance.y, radiance.z, __uint_as_float(seed)));
}

template <bool BINARY, int CAP, bool STREAM>
__global__ void __launch_bounds__(128)
render_mega_kernel(SceneView s, FrameArgs a, float* __restrict__ result, GidMap map, uint32_t n, RadianceIO io) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t g = map.gid(i);
    uint32_t seed;
    RayX r;
    float tmax = 100000.0f;                                               // segment 0 of a frame: kernel_bvh.cl:355
    if (STREAM) {
        float4 q0, q1;
        stream_path_start(io, g, q0, q1, seed);
        r = make_ray(q0.x, q0.y, q0.z, q1.x, q1.y, q1.z);
        tmax = q1.w;
    } else {
        uint32_t gid = (uint32_t)g;
        seed = gid + hash_u32(a.frame_count);                             // kernel_bvh.cl:445
        V3 dir = camera_dir(a, gid, seed);
        r = make_ray(a.pos[0], a.pos[1], a.pos[2], dir.x, dir.y, dir.z);
    }
    V3 radiance = v3(0.0f, 0.0f, 0.0f), beta = v3(1.0f, 1.0f, 1.0f);
    for (int b = 0; (uint32_t)b < (uint32_t)a.bounces; ++b) {              // Render(), kernel_bvh.cl:349-384
        HitX h;
        if (BINARY) h = trace_binary<false, CAP>(s.tris, s.nodes, r, tmax);
        else h = trace_wide<false, false, CAP>(s.wide, s.leaf, r, tmax, nullptr, nullptr, s.one_bits);
        V3 no, nd;
        if (!path_step(s, a, r, h, radiance, beta, seed, no, nd)) break;
        r = make_ray(no.x, no.y, no.z, nd.x, nd.y, nd.z);
        if (STREAM) tmax = 100000.0f;
    }
    radiance = v3(max_cl(radiance.x, 0.0f), max_cl(radiance.y, 0.0f), max_cl(radiance.z, 0.0f));
    if (STREAM) store_radiance(io, g, radiance, seed);
    else accumulate(result + 4 * g, a.mirror ? a.mirror + 4 * g : nullptr, radiance, a.frame_count);
}

// ---------------------------------------------------------------------------------------
// Wavefront frame path: generate -> { trace_persistent -> shade } x lightBounces.
//
// Path i of the shard keeps {radiance, seed | beta} in state[2i], state[2i+1]; the ray queues hold
// b2rt_ray records whose (ignored) tmin slot carries i, so only the 32-byte ray is compacted between
// bounces. Hits are written by trace_persistent at the ray's queue position. Every path runs the same
// arithmetic in the same order as KernelEntry, so frames are bit-identical to the megakernel's.
// STREAM = true: the same stages for a caller's ray stream (b2rt_trace_radiance, see render_mega_kernel).
// ---------------------------------------------------------------------------------------
template <bool STREAM>
__global__ void __launch_bounds__(256)
wf_generate_kernel(FrameArgs a, GidMap map, uint32_t n, RayIn* __restrict__ rays, float4* __restrict__ state,
                   unsigned long long* __restrict__ queue_count, RadianceIO io) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    // counter block of this wavefront: [0..2] rotating queue lengths, [3] the traversal kernel's ray counter, [4] [5] its tail queue's length and read position, [6] [7] the second tail queue's, [8] [9] [10] helping: warps past their hand-over, warps started, tickets given back
    if (i == 0) { queue_count[0] = n; for (int k = 1; k < 16; ++k) queue_count[k] = 0; }
    if (i >= n) return;
    uint32_t seed;
    float4 q0, q1;
    if (STREAM) {
        stream_path_start(io, map.gid(i), q0, q1, seed);                  // the direction as given and the caller's tmax
    } else {
        uint32_t gid = (uint32_t)map.gid(i);
        seed = gid + hash_u32(a.frame_count);                             // kernel_bvh.cl:445
        V3 d = camera_dir(a, gid, seed);
        q0 = make_float4(a.pos[0], a.pos[1], a.pos[2], 0.0f);
        q1 = make_float4(d.x, d.y, d.z, 100000.0f);                       // InitRay normalises again inside the trace stage
    }
    float4* p = reinterpret_cast<float4*>(rays + i);
    p[0] = make_float4(q0.x, q0.y, q0.z, __uint_as_float(i));
    p[1] = q1;
    state[2 * (size_t)i] = make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(seed));
    state[2 * (size_t)i + 1] = make_float4(1.0f, 1.0f, 1.0f, 0.0f);
}

template <bool STREAM>
__global__ void __launch_bounds__(256)
wf_shade_kernel(SceneView s, FrameArgs a, GidMap map, const RayIn* __restrict__ rays_in, const float4* __restrict__ hits,
                const unsigned long long* __restrict__ n_in, RayIn* __restrict__ rays_out,
                unsigned long long* __restrict__ n_out, float4* __restrict__ state, float* __restrict__ result, int last,
                unsigned long long* __restrict__ clear_a, unsigned long long* __restrict__ clear_b, RadianceIO io) {
    const uint64_t n = *n_in;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    // reset what the NEXT stages start from: the traversal kernel's ray counter and the queue length the next
    // shade stage appends to (neither is read or written by anything in flight now)
    if (j == 0) { *clear_a = 0; for (int k = 0; k < 8; ++k) clear_b[k] = 0; }
    if ((j & ~31ull) >= n) return;                      // whole warp beyond the queue
    const unsigned lane = threadIdx.x & 31u;
    bool go_on = false;
    uint32_t i = 0;
    RayX r;
    V3 radiance, beta, no, nd;
    uint32_t seed = 0;
    if (j < n) {
        const float4* p = reinterpret_cast<const float4*>(rays_in + j);
        float4 q0 = __ldg(p), q1 = __ldg(p + 1);
        i = __float_as_uint(q0.w);
        r = make_ray(q0.x, q0.y, q0.z, q1.x, q1.y, q1.z);
        float4 hv = __ldg(hits + j);
        HitX h; h.t = hv.x; h.u = hv.y; h.v = hv.z; h.tri = __float_as_uint(hv.w);
        float4 s0 = state[2 * (size_t)i], s1 = state[2 * (size_t)i + 1];
        radiance = v3(s0.x, s0.y, s0.z); seed = __float_as_uint(s0.w);
        beta = v3(s1.x, s1.y, s1.z);
        go_on = path_step(s, a, r, h, radiance, beta, seed, no, nd) && !last;
        if (!go_on) {
            radiance = v3(max_cl(radiance.x, 0.0f), max_cl(radiance.y, 0.0f), max_cl(radiance.z, 0.0f));
            const uint64_t g = map.gid(i);
            if (STREAM) store_radiance(io, g, radiance, seed);
            else accumulate(result + 4 * g, a.mirror ? a.mirror + 4 * g : nullptr, radiance, a.frame_count);
        }
    }
    // append the surviving rays to the next queue: one atomic per warp
    const unsigned m = __ballot_sync(FULL, go_on);
    if (m == 0u) return;
    unsigned long long base = 0;
    const unsigned leader = __ffs(m) - 1;
    if (lane == leader) base = atomicAdd(n_out, (unsigned long long)__popc(m));
    base = __shfl_sync(FULL, base, leader);
    if (go_on) {
        const uint64_t slot = base + __popc(m & ((1u << lane) - 1u));
        float4* p = reinterpret_cast<float4*>(rays_out + slot);
        // the queue carries InitRay's arguments; the trace stage (and the next shade stage) normalise them
        // exactly once, like the megakernel's make_ray(no, wi)
        p[0] = make_float4(no.x, no.y, no.z, __uint_as_float(i));
        p[1] = make_float4(nd.x, nd.y, nd.z, 100000.0f);
        state[2 * (size_t)i] = make_float4(radiance.x, radiance.y, radiance.z, __uint_as_float(seed));
        state[2 * (size_t)i + 1] = make_float4(beta.x, beta.y, beta.z, 0.0f);
    }
}

// ---------------------------------------------------------------------------------------
// Output path (SURVEY.md 8f-4): the accumulation image already holds display-referred (gamma 1/2.2) values
// (kernel_bvh.cl:449-455) which the reference reads back as 16 B/pixel and re-uploads to GL as GL_RGBA/GL_FLOAT
// (CLRaytracer.cpp:55,64-67), i.e. GL clamps them to [0,1] for an 8-bit target. This kernel does that clamp and
// the 8-bit quantisation on the device so that only 4 B/pixel cross PCIe. NaN -> 0 (saturate), alpha = 255.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
tonemap_rgba8_kernel(const float4* __restrict__ image, uchar4* __restrict__ out, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = image[i];
    out[i] = make_uchar4((unsigned char)__float2uint_rn(__saturatef(p.x) * 255.0f), (unsigned char)__float2uint_rn(__saturatef(p.y) * 255.0f),
                         (unsigned char)__float2uint_rn(__saturatef(p.z) * 255.0f), 255);
}

// ---------------------------------------------------------------------------------------
// Closest point (b2rt_closest_point). Every lane owns one query (PointLane, point_query.cuh); warps pull chunks of queries
// from a global atomic counter into a warp-local pool and refill idle lanes from it (ballot + popc compaction), like
// trace_persistent. Per round the warp votes: the lanes that want a wide-node step or those that want a leaf step, by
// majority. The result does not depend on the schedule: it is the minimum of the total order (d2, tri).
// ---------------------------------------------------------------------------------------
static constexpr int POINT_BLOCK = 128;

__device__ __forceinline__ void write_point(float4* __restrict__ out, uint64_t i, const PointHit& h) {
    __stcs(out + i, make_float4(h.d2, h.u, h.v, __uint_as_float(h.tri)));
}

template <bool COUNT, int CAP>
__global__ void __launch_bounds__(POINT_BLOCK, B2_MIN_BLOCKS)
point_persistent(SceneView s, const float4* __restrict__ queries, uint64_t n, float4* __restrict__ out,
                 unsigned long long* __restrict__ next, unsigned long long* __restrict__ counters, uint32_t chunk, uint32_t refill_min) {
    const unsigned lane = threadIdx.x & 31u;
    PointLane<COUNT, CAP> L;
    PointEntry stack[CAP];
    L.cur = REF_EMPTY; L.sp = 0; L.overflow = false;
    L.tc.wide_nodes = L.tc.leaf_blocks = L.tc.tri_tests = L.tc.words = L.tc.max_stack = 0;
    uint64_t my_index = 0, pool_next = 0;
    uint32_t pool_left = 0, started = 0;
    bool dry = false;                        // warp-uniform: the global counter has run past n
    for (;;) {
        const unsigned vn = __ballot_sync(FULL, L.wants_node());
        const unsigned vl = __ballot_sync(FULL, L.wants_leaf());
        const unsigned busy = vn | vl;
        if (32u - (unsigned)__popc(busy) >= (dry ? 32u : refill_min)) {
            if (dry) break;
            if (pool_left == 0u) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(next, (unsigned long long)chunk);
                base = __shfl_sync(FULL, base, 0);
                if (base >= n) { dry = true; continue; }
                pool_next = base;
                pool_left = (base + chunk < n) ? chunk : (uint32_t)(n - base);
            }
            const unsigned idle = ~busy;
            const unsigned rank = __popc(idle & ((1u << lane) - 1u));
            if (((idle >> lane) & 1u) && rank < pool_left) {
                my_index = pool_next + rank;
                const float4 q = __ldcs(queries + my_index);
                if (!L.start(q.x, q.y, q.z, q.w)) write_point(out, my_index, L.best);      // misses without a walk
                if (COUNT) started++;
            }
            const unsigned taken = __popc(idle), used = taken < pool_left ? taken : pool_left;
            pool_next += used;
            pool_left -= used;
            continue;
        }
        bool stepped;
        if (__popc(vn) >= __popc(vl)) { stepped = L.wants_node(); if (stepped) L.node_step(s.wide, stack); }
        else { stepped = L.wants_leaf(); if (stepped) L.leaf_step(s.leaf, stack); }
        if (stepped && L.done()) write_point(out, my_index, L.best);
    }
    if (COUNT) {
        if (L.overflow) report_stack_overflow();
        // the ray counters' slots: [0] queries, [1] wide-node visits, [2] leaf blocks, [4] distance evaluations, [5] words
        unsigned long long v[5] = { started, L.tc.wide_nodes, L.tc.leaf_blocks, L.tc.tri_tests, L.tc.words };
        const int slot[5] = { 0, 1, 2, 4, 5 };
#pragma unroll
        for (int i = 0; i < 5; ++i) {
            unsigned long long x = v[i];
            for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(FULL, x, o);
            if (lane == 0 && x) atomicAdd(&counters[slot[i]], x);
        }
    }
}

// The same query over the reference's CLLinearBVHNode / CLTriangle arrays, one thread per query: a node is entered iff the
// lb of its exact fp32 box is <= the best so far; the child on the point's side of the box's middle goes first. The stack
// holds one entry per level (CAP >= max_depth_binary, as for trace_binary).
template <int CAP>
__global__ void __launch_bounds__(128)
point_binary_kernel(SceneView s, const float4* __restrict__ queries, uint64_t n, float4* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 q = __ldg(queries + i);
    PointHit best; best.d2 = q.w; best.u = 0.0f; best.v = 0.0f; best.tri = 0xFFFFFFFFu;
    if (q.x == q.x && q.y == q.y && q.z == q.z && q.w >= 0.0f) {
        uint32_t stack[CAP];
        int sp = 0;
        uint32_t cur = 0;
        for (;;) {
            const float4* np = reinterpret_cast<const float4*>(s.nodes + cur);
            const float4 lo = __ldg(np), hi = __ldg(np + 1);
            const uint4 tail = __ldg(reinterpret_cast<const uint4*>(np + 2));
            const uint32_t nprim = tail.y & 0xffffu, axis = (tail.y >> 16) & 0xffu;
            bool descend = false;
            if (box_lb(q.x, q.y, q.z, lo.x, lo.y, lo.z, hi.x, hi.y, hi.z) <= best.d2) {
                if (nprim > 0) {
                    for (uint32_t k = 0; k < nprim; ++k) {
                        const float4* tp = reinterpret_cast<const float4*>(s.tris + tail.x + k);
                        const float4 a = __ldg(tp), b = __ldg(tp + 5), c = __ldg(tp + 10);   // positions at +0, +80, +160 B
                        float d2, u, v;
                        closest_on_triangle(q.x, q.y, q.z, a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z, d2, u, v);
                        point_take(best, d2, u, v, tail.x + k);
                    }
                } else {
                    descend = true;
                    const float pa = axis == 0 ? q.x : (axis == 1 ? q.y : q.z);
                    const float mid = axis == 0 ? xadd(lo.x, hi.x) : (axis == 1 ? xadd(lo.y, hi.y) : xadd(lo.z, hi.z));
                    const bool second_first = xadd(pa, pa) > mid;
                    if (sp < CAP) stack[sp++] = second_first ? cur + 1u : tail.x;
                    else report_stack_overflow();
                    cur = second_first ? tail.x : cur + 1u;
                }
            }
            if (!descend) {
                if (sp == 0) break;
                cur = stack[--sp];
            }
        }
    }
    out[i] = make_float4(best.d2, best.u, best.v, __uint_as_float(best.tri));
}

// ---------------------------------------------------------------------------------------
// Launch wrappers (host).
// ---------------------------------------------------------------------------------------
static int pick_cap(uint32_t bound) { return bound <= 32 ? 32 : (bound <= 64 ? 64 : (bound <= 128 ? 128 : (bound <= 256 ? 256 : 0))); }

// Calls f(std::integral_constant<int, CAP>()) for the smallest stack capacity CAP that holds `bound` entries, then returns
// the launch status; a bound past 256 has no kernel and returns cudaErrorInvalidValue.
template <class F>
static cudaError_t with_cap(uint32_t bound, F&& f) {
    switch (pick_cap(bound)) {
        case 32: f(std::integral_constant<int, 32>()); break;
        case 64: f(std::integral_constant<int, 64>()); break;
        case 128: f(std::integral_constant<int, 128>()); break;
        case 256: f(std::integral_constant<int, 256>()); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// Pool scheduling of the persistent kernels: items per pool top-up, about 1/8 of a warp's fair share, a multiple of 32
// in [32, 512] ...
static uint32_t pool_chunk(uint64_t n, int grid, int block) {
    const uint64_t warps = (uint64_t)grid * (block / 32), c = n / (warps * 8u + 1u);
    return (uint32_t)(c < 32 ? 32 : (c > 512 ? 512 : (c & ~31ull)));
}
// ... and the idle lanes that trigger a refill, 8 when out of range
static uint32_t refill_or_default(uint32_t refill_min) { return (refill_min < 1 || refill_min > 32) ? 8u : refill_min; }

template <int P, bool COUNT>
static cudaError_t launch_persistent(uint32_t stack_bound, int grid, cudaStream_t st, const SceneView& s, const void* rays,
                                     uint64_t n, void* out, unsigned long long* next, unsigned long long* counters,
                                     uint32_t refill_min, uint32_t leaf_bias, const unsigned long long* n_dev, const TailQueue& tail,
                                     const uint32_t* resume = nullptr, uint32_t k = 0) {
    const RayIn* r = static_cast<const RayIn*>(rays);
    const uint32_t chunk = pool_chunk(n, grid, TRACE_BLOCK);
    refill_min = refill_or_default(refill_min);
    if (leaf_bias < 1 || leaf_bias > 512) leaf_bias = 16;
    return with_cap(stack_bound, [&](auto C) {
        trace_persistent<P, COUNT, C><<<grid, TRACE_BLOCK, 0, st>>>(s, r, n, out, next, counters, chunk, refill_min, leaf_bias, n_dev, tail, resume, k);
    });
}

cudaError_t launch_trace_wide(const SceneView& s, const void* d_rays, uint64_t n, void* d_out, bool any, bool count,
                              uint32_t stack_bound, int grid_blocks, unsigned long long* d_next,
                              unsigned long long* d_counters, uint32_t refill_min, uint32_t leaf_bias, cudaStream_t st,
                              const unsigned long long* d_n, const TailQueue* tail_in, int tail_grid, cudaEvent_t between) {
    if (!pick_cap(stack_bound)) return cudaErrorInvalidValue;
    TailQueue tail = { nullptr, nullptr, nullptr, 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0 };
    if (tail_in && tail_in->coop_max && tail_in->records) tail = *tail_in;
    const bool two_step = tail.coop_max && tail.resume_max && tail.records2;
    if (!d_n) {     // wavefront stages (d_n given) get their counters reset by the preceding stage's kernel
        // [0] the ray counter, [1] [2] tail-queue length and read position, [3] [4] the second tail queue's, [5] [6] [7] helping: warps past their hand-over, warps started, tickets given back
        cudaError_t e = cudaMemsetAsync(d_next, 0, 8 * sizeof(unsigned long long), st);
        if (e != cudaSuccess) return e;
    }
    // what each pass hands over to: the first pass suspends into queue 1 (at resume_max live rays when a second pass follows)
    // helping: only when the helping warp's shared memory holds the tail kernel's frontier, and not in the two-step mode (its
    // first queue is the second pass's ray stream)
    const uint32_t fcap_tail = tail_frontier_words(stack_bound);
    if (two_step || !tail.help_fcap || !tail.handed || !tail.orphans || !tail.tag || fcap_tail > trace_warp_smem_words()) tail.help_fcap = 0;
    else { tail.help_fcap = fcap_tail; tail.help_wide_limit = fcap_tail - (stack_bound + 8u) - (7u * B2_COOP_NODES + 4u); }
    TailQueue q1 = tail;
    if (two_step) q1.coop_max = tail.resume_max;
    TailQueue q2 = tail;
    if (two_step) { q2.count = tail.count2; q2.next = tail.next2; q2.records = tail.records2; }
    auto pass = [&](const unsigned long long* n_dev, unsigned long long* next, const TailQueue& q, const uint32_t* resume) -> cudaError_t {
        if (any) return count ? launch_persistent<HIT_ANY, true>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, next, d_counters, refill_min, leaf_bias, n_dev, q, resume)
                              : launch_persistent<HIT_ANY, false>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, next, d_counters, refill_min, leaf_bias, n_dev, q, resume);
        return count ? launch_persistent<HIT_CLOSEST, true>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, next, d_counters, refill_min, leaf_bias, n_dev, q, resume)
                     : launch_persistent<HIT_CLOSEST, false>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, next, d_counters, refill_min, leaf_bias, n_dev, q, resume);
    };
    cudaError_t e = pass(d_n, d_next, q1, nullptr);
    // second pass: the suspended rays are its ray stream (count and read position = queue 1's counters)
    if (e == cudaSuccess && two_step) e = pass(tail.count, tail.next, q2, tail.records);
    if (e == cudaSuccess && between) e = cudaEventRecord(between, st);
    if (e != cudaSuccess || !tail.coop_max) return e;
    // the tail kernel: frontier capacity per warp and the size up to which four nodes are expanded per round
    const uint32_t fcap = tail_frontier_words(stack_bound), wide_limit = fcap - (stack_bound + 8u) - (7u * B2_COOP_NODES + 4u);   // a round adds at most 7 entries per expanded node
    const size_t smem = (size_t)(TAIL_BLOCK / 32) * fcap * sizeof(uint32_t);
    const RayIn* r = static_cast<const RayIn*>(d_rays);
    if (any) { if (count) trace_tail_kernel<true, true><<<tail_grid, TAIL_BLOCK, smem, st>>>(s, r, d_out, q2, d_counters, fcap, wide_limit);
               else trace_tail_kernel<true, false><<<tail_grid, TAIL_BLOCK, smem, st>>>(s, r, d_out, q2, d_counters, fcap, wide_limit); }
    else { if (count) trace_tail_kernel<false, true><<<tail_grid, TAIL_BLOCK, smem, st>>>(s, r, d_out, q2, d_counters, fcap, wide_limit);
           else trace_tail_kernel<false, false><<<tail_grid, TAIL_BLOCK, smem, st>>>(s, r, d_out, q2, d_counters, fcap, wide_limit); }
    return cudaGetLastError();
}

cudaError_t launch_trace_multi(const SceneView& s, const void* d_rays, uint64_t n, uint32_t k, void* d_out, bool count,
                               uint32_t stack_bound, int grid_blocks, unsigned long long* d_next, unsigned long long* d_counters,
                               uint32_t refill_min, uint32_t leaf_bias, cudaStream_t st) {
    if (!pick_cap(stack_bound) || k == 0) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(d_next, 0, 8 * sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    const TailQueue none = { nullptr, nullptr, nullptr, 0, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, 0 };
    return count ? launch_persistent<HIT_MULTI, true>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, d_next, d_counters, refill_min, leaf_bias, nullptr, none, nullptr, k)
                 : launch_persistent<HIT_MULTI, false>(stack_bound, grid_blocks, st, s, d_rays, n, d_out, d_next, d_counters, refill_min, leaf_bias, nullptr, none, nullptr, k);
}

uint32_t trace_warp_smem_words() { return (B2_TAIL_HELP && B2_TAIL_CODE) ? (uint32_t)WARP_SMEM_WORDS : 0u; }
uint32_t tail_frontier_words(uint32_t stack_bound) { uint32_t w = 4u * (stack_bound + 8u); return w < 256u ? 256u : w; }
uint32_t tail_record_words(uint32_t stack_bound) { return TAIL_HEADER_WORDS + ((stack_bound + 8u + 3u) & ~3u); }

cudaError_t launch_trace_binary(const SceneView& s, const void* d_rays, uint64_t n, void* d_out, bool any, uint32_t max_depth_binary,
                                cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    uint64_t blocks = (n + 127) / 128;
    if (blocks > 0x7fffffffull) return cudaErrorInvalidValue;
    const RayIn* r = static_cast<const RayIn*>(d_rays);
    return with_cap(max_depth_binary, [&](auto C) {
        if (any) trace_binary_kernel<true, C><<<(unsigned)blocks, 128, 0, st>>>(s, r, n, d_out);
        else trace_binary_kernel<false, C><<<(unsigned)blocks, 128, 0, st>>>(s, r, n, d_out);
    });
}

cudaError_t launch_trace_binary_multi(const SceneView& s, const void* d_rays, uint64_t n, uint32_t k, void* d_out, uint32_t max_depth_binary,
                                      cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    uint64_t blocks = (n + 127) / 128;
    if (blocks > 0x7fffffffull || k == 0) return cudaErrorInvalidValue;
    const RayIn* r = static_cast<const RayIn*>(d_rays);
    HitX* out = static_cast<HitX*>(d_out);
    return with_cap(max_depth_binary, [&](auto C) { trace_binary_multi_kernel<C><<<(unsigned)blocks, 128, 0, st>>>(s, r, n, out, k); });
}

cudaError_t launch_camera_rays(const FrameArgs& a, uint64_t gid0, uint64_t gid1, void* d_rays, cudaStream_t st) {
    if (gid1 <= gid0) return cudaSuccess;
    uint64_t blocks = (gid1 - gid0 + 255) / 256;
    if (blocks > 0x7fffffffull) return cudaErrorInvalidValue;
    camera_rays_kernel<<<(unsigned)blocks, 256, 0, st>>>(a, gid0, gid1, static_cast<RayIn*>(d_rays));
    return cudaGetLastError();
}

cudaError_t launch_render_mega(const SceneView& s, const FrameArgs& a, float* d_result, const GidMap& map, uint32_t n,
                               bool binary, uint32_t stack_bound, uint32_t max_depth_binary, cudaStream_t st, const RadianceIO* io) {
    if (n == 0) return cudaSuccess;
    unsigned g = (n + 127u) / 128u;
    // the wide walk holds at most stack_bound entries, the reference-layout walk at most max_depth_binary
    return with_cap(binary ? max_depth_binary : stack_bound, [&](auto C) {
        if (io) {
            if (binary) render_mega_kernel<true, C, true><<<g, 128, 0, st>>>(s, a, nullptr, map, n, *io);
            else render_mega_kernel<false, C, true><<<g, 128, 0, st>>>(s, a, nullptr, map, n, *io);
        } else {
            if (binary) render_mega_kernel<true, C, false><<<g, 128, 0, st>>>(s, a, d_result, map, n, RadianceIO{ nullptr, nullptr, nullptr });
            else render_mega_kernel<false, C, false><<<g, 128, 0, st>>>(s, a, d_result, map, n, RadianceIO{ nullptr, nullptr, nullptr });
        }
    });
}

cudaError_t launch_wf_generate(const FrameArgs& a, const GidMap& map, uint32_t n, void* d_rays, void* d_state,
                               unsigned long long* d_queue_count, cudaStream_t st, const RadianceIO* io) {
    if (n == 0) return cudaSuccess;
    RayIn* rays = static_cast<RayIn*>(d_rays);
    float4* state = static_cast<float4*>(d_state);
    if (io) wf_generate_kernel<true><<<(n + 255u) / 256u, 256, 0, st>>>(a, map, n, rays, state, d_queue_count, *io);
    else wf_generate_kernel<false><<<(n + 255u) / 256u, 256, 0, st>>>(a, map, n, rays, state, d_queue_count, RadianceIO{ nullptr, nullptr, nullptr });
    return cudaGetLastError();
}

cudaError_t launch_wf_shade(const SceneView& s, const FrameArgs& a, const GidMap& map, uint32_t n_max, const void* d_rays_in,
                            const void* d_hits, const unsigned long long* d_n_in, void* d_rays_out, unsigned long long* d_n_out,
                            void* d_state, float* d_result, bool last, unsigned long long* d_clear_a, unsigned long long* d_clear_b,
                            cudaStream_t st, const RadianceIO* io) {
    if (n_max == 0) return cudaSuccess;
    const unsigned g = (n_max + 255u) / 256u;
    const RayIn* in = static_cast<const RayIn*>(d_rays_in);
    const float4* hits = static_cast<const float4*>(d_hits);
    RayIn* out = static_cast<RayIn*>(d_rays_out);
    float4* state = static_cast<float4*>(d_state);
    if (io) wf_shade_kernel<true><<<g, 256, 0, st>>>(s, a, map, in, hits, d_n_in, out, d_n_out, state, nullptr, last ? 1 : 0, d_clear_a, d_clear_b, *io);
    else wf_shade_kernel<false><<<g, 256, 0, st>>>(s, a, map, in, hits, d_n_in, out, d_n_out, state, d_result, last ? 1 : 0, d_clear_a, d_clear_b,
                                                    RadianceIO{ nullptr, nullptr, nullptr });
    return cudaGetLastError();
}

cudaError_t launch_tonemap_rgba8(const void* d_image, void* d_out, uint64_t n, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    uint64_t blocks = (n + 255) / 256;
    if (blocks > 0x7fffffffull) return cudaErrorInvalidValue;
    tonemap_rgba8_kernel<<<(unsigned)blocks, 256, 0, st>>>(static_cast<const float4*>(d_image), static_cast<uchar4*>(d_out), n);
    return cudaGetLastError();
}

cudaError_t launch_closest_point(const SceneView& s, const void* d_queries, uint64_t n, void* d_out, bool count, uint32_t stack_bound,
                                 int grid_blocks, unsigned long long* d_next, unsigned long long* d_counters, uint32_t refill_min,
                                 cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    if (!pick_cap(stack_bound) || grid_blocks < 1) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(d_next, 0, sizeof(unsigned long long), st);
    if (e != cudaSuccess) return e;
    refill_min = refill_or_default(refill_min);
    const uint32_t chunk = pool_chunk(n, grid_blocks, POINT_BLOCK);
    const float4* q = static_cast<const float4*>(d_queries);
    float4* out = static_cast<float4*>(d_out);
    return with_cap(stack_bound, [&](auto C) {
        if (count) point_persistent<true, C><<<grid_blocks, POINT_BLOCK, 0, st>>>(s, q, n, out, d_next, d_counters, chunk, refill_min);
        else point_persistent<false, C><<<grid_blocks, POINT_BLOCK, 0, st>>>(s, q, n, out, d_next, d_counters, chunk, refill_min);
    });
}

cudaError_t launch_closest_point_binary(const SceneView& s, const void* d_queries, uint64_t n, void* d_out, uint32_t max_depth_binary,
                                        cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const uint64_t blocks = (n + 127) / 128;
    if (blocks > 0x7fffffffull) return cudaErrorInvalidValue;
    const float4* q = static_cast<const float4*>(d_queries);
    float4* out = static_cast<float4*>(d_out);
    return with_cap(max_depth_binary, [&](auto C) { point_binary_kernel<C><<<(unsigned)blocks, 128, 0, st>>>(s, q, n, out); });
}

int trace_block_threads() { return TRACE_BLOCK; }

cudaError_t stack_overflow_count(unsigned long long* out, bool reset) {
    cudaError_t e = cudaSuccess;
    if (out) e = cudaMemcpyFromSymbol(out, g_stack_overflows, sizeof(unsigned long long));
    if (e == cudaSuccess && reset) { const unsigned long long zero = 0; e = cudaMemcpyToSymbol(g_stack_overflows, &zero, sizeof(zero)); }
    return e;
}

cudaError_t tail_occupancy(uint32_t stack_bound, int* blocks_per_sm) {
    const size_t smem = (size_t)(TAIL_BLOCK / 32) * tail_frontier_words(stack_bound) * sizeof(uint32_t);
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, trace_tail_kernel<false, false>, TAIL_BLOCK, smem);
}

cudaError_t trace_occupancy(bool any, uint32_t stack_bound, int* blocks_per_sm) {
    const void* fn = nullptr;
    cudaError_t e = with_cap(stack_bound, [&](auto C) {
        fn = any ? (const void*)trace_persistent<HIT_ANY, false, C> : (const void*)trace_persistent<HIT_CLOSEST, false, C>;
    });
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, TRACE_BLOCK, 0);
}

}  // namespace b2rt
