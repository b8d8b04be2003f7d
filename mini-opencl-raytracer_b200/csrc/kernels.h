// kernels.h -- host-callable launch wrappers implemented in kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "b2rt_types.h"

namespace b2rt {

// Tail queue of a persistent traversal launch (see trace_tail_kernel in kernels.cu). coop_max = 0 switches the tail mode off.
struct TailQueue {
    unsigned long long* count;     // records written by the launch (device counter, zeroed before it)
    unsigned long long* next;      // read position of the tail kernel (zeroed likewise)
    uint32_t* records;             // capacity: coop_max records per warp of the persistent grid
    uint32_t rec_words;            // tail_record_words(stack_bound)
    uint32_t coop_max;             // a dry warp with at most this many live rays hands them over
    // Two-step tail (resume_max > 0): the persistent launch suspends at resume_max live rays per dry warp into THIS queue,
    // a second persistent launch re-packs the suspended rays 32 to a warp and walks on (full SIMT width again), hands what
    // is left at coop_max live rays per warp to the second queue below, and the cooperative kernel finishes those.
    uint32_t resume_max;
    unsigned long long* count2;
    unsigned long long* next2;
    uint32_t* records2;
    // Helping (help_fcap > 0): a warp of the persistent launch that has handed its last rays over serves the queue itself
    // (trace_persistent's epilogue) while other warps are still walking; what is left when the launch ends goes to the tail
    // kernel as before. `handed` counts the warps that are past their hand-over (zeroed with the other counters), `tag`
    // (unique per launch, never 0) marks a record as completely written.
    unsigned long long* handed;    // [0] warps past their hand-over, [1] warps started, [2] tickets in `orphans`
    unsigned long long* orphans;   // tickets (queue positions) that helping warps drew and gave back: one per warp of the grid at most
    uint32_t tag;
    uint32_t help_fcap;            // frontier words a helping warp has (its own shared-memory columns); 0 = no helping
    uint32_t help_wide_limit;      // frontier size up to which a helping warp expands several nodes per round (as in the tail kernel)
};
uint32_t trace_warp_smem_words();                     // shared-memory words each warp of trace_persistent owns
uint32_t tail_frontier_words(uint32_t stack_bound);   // shared-memory words per warp of the tail kernel
uint32_t tail_record_words(uint32_t stack_bound);

// Persistent while-while traversal of the compressed wide BVH over a device-resident ray
// stream. d_out is b2rt_hit[n] (closest) or uint32_t[n] (any). d_next points at five 64-bit scratch
// counters (ray counter, tail-queue length and read position, second tail queue's likewise; reset by the wrapper unless d_n is given),
// d_counters twenty-four 64-bit accumulators (used when count; [13] = stack/frontier overflows, always). With a tail
// queue the cooperative tail kernel is launched right behind the persistent one (tail_grid blocks).
cudaError_t launch_trace_wide(const SceneView& s, const void* d_rays, uint64_t n, void* d_out, bool any, bool count,
                              uint32_t stack_bound, int grid_blocks, unsigned long long* d_next,
                              unsigned long long* d_counters, uint32_t refill_min, uint32_t leaf_bias, cudaStream_t st,
                              const unsigned long long* d_n = nullptr,    // d_n != null: ray count read on the device (n = upper bound)
                              const TailQueue* tail = nullptr, int tail_grid = 0,
                              cudaEvent_t between = nullptr);           // recorded between the persistent and the tail kernel (stage timing)
// One thread per ray over the reference-layout arrays (baseline / cross-check). Its stack holds max_depth_binary entries
// (b2rt_scene_info); cudaErrorInvalidValue for a tree deeper than 256 levels.
cudaError_t launch_trace_binary(const SceneView& s, const void* d_rays, uint64_t n, void* d_out, bool any, uint32_t max_depth_binary,
                                cudaStream_t st);
// The k nearest hits per ray (1 <= k): d_out is b2rt_hit[n * k], row i sorted by t and padded with misses. The persistent
// kernel with the HIT_MULTI policy, without a cooperative tail (d_next: eight 64-bit scratch counters, reset here) ...
cudaError_t launch_trace_multi(const SceneView& s, const void* d_rays, uint64_t n, uint32_t k, void* d_out, bool count,
                               uint32_t stack_bound, int grid_blocks, unsigned long long* d_next, unsigned long long* d_counters,
                               uint32_t refill_min, uint32_t leaf_bias, cudaStream_t st);
// ... and the same over the reference-layout arrays, one thread per ray.
cudaError_t launch_trace_binary_multi(const SceneView& s, const void* d_rays, uint64_t n, uint32_t k, void* d_out, uint32_t max_depth_binary,
                                      cudaStream_t st);
// Closest point per query (b2rt_closest_point): d_queries = b2rt_point_query[n], d_out = b2rt_point_hit[n]. The persistent
// kernel over the compressed wide BVH (d_next: one 64-bit scratch counter, reset here) ...
cudaError_t launch_closest_point(const SceneView& s, const void* d_queries, uint64_t n, void* d_out, bool count, uint32_t stack_bound,
                                 int grid_blocks, unsigned long long* d_next, unsigned long long* d_counters, uint32_t refill_min,
                                 cudaStream_t st);
// ... and the same over the reference-layout arrays, one thread per query.
cudaError_t launch_closest_point_binary(const SceneView& s, const void* d_queries, uint64_t n, void* d_out, uint32_t max_depth_binary,
                                        cudaStream_t st);
cudaError_t launch_camera_rays(const FrameArgs& a, uint64_t gid0, uint64_t gid1, void* d_rays, cudaStream_t st);
// A caller's ray stream as the source and sink of the frame kernels below (b2rt_trace_radiance): the path of work item g =
// map.gid(i) starts from rays[g] (b2rt_ray) with RNG state seeds[g], and out[g] (b2rt_radiance) receives its record. Only
// bounces, light_type and sky of the FrameArgs are read then, and d_result is not used.
struct RadianceIO {
    const void* rays;
    const uint32_t* seeds;
    void* out;
};
// KernelEntry for the n pixels map.gid(0..n-1), one thread per pixel; binary: over the reference-layout arrays.
cudaError_t launch_render_mega(const SceneView& s, const FrameArgs& a, float* d_result, const GidMap& map, uint32_t n,
                               bool binary, uint32_t stack_bound, uint32_t max_depth_binary, cudaStream_t st, const RadianceIO* io = nullptr);
// Wavefront stages of the same frame (kernels.cu): camera rays + path state, and the per-bounce shade/compact stage.
cudaError_t launch_wf_generate(const FrameArgs& a, const GidMap& map, uint32_t n, void* d_rays, void* d_state,
                               unsigned long long* d_queue_count, cudaStream_t st, const RadianceIO* io = nullptr);
cudaError_t launch_wf_shade(const SceneView& s, const FrameArgs& a, const GidMap& map, uint32_t n_max, const void* d_rays_in,
                            const void* d_hits, const unsigned long long* d_n_in, void* d_rays_out, unsigned long long* d_n_out,
                            void* d_state, float* d_result, bool last, unsigned long long* d_clear_a, unsigned long long* d_clear_b,
                            cudaStream_t st, const RadianceIO* io = nullptr);
// float4 accumulation image -> clamped 8-bit RGBA (alpha 255), n pixels.
cudaError_t launch_tonemap_rgba8(const void* d_image, void* d_out, uint64_t n, cudaStream_t st);
int trace_block_threads();
// Stack / frontier overflows seen by the traversal kernels on the current device since the last reset (never expected).
cudaError_t stack_overflow_count(unsigned long long* out, bool reset);
cudaError_t tail_occupancy(uint32_t stack_bound, int* blocks_per_sm);
cudaError_t trace_occupancy(bool any, uint32_t stack_bound, int* blocks_per_sm);

}  // namespace b2rt
