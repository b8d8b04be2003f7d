// context.h -- internal: the state behind a b2rt_context handle and the helpers shared by api.cu (single-device entry
// points) and multi.cu (device groups, NCCL, peer-mapped frame gather). Not installed; include/b2rt.h is the interface.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>
#include "b2rt.h"
#include "kernels.h"

namespace b2rt_detail {

struct Buffer {
    void* d_ptr = nullptr;
    size_t bytes = 0;
    uint32_t flags = 0;
    std::vector<uint8_t> shadow;   // host copy of COPY_HOST_PTR data, dropped once the wide BVH is built
};

constexpr uint64_t STREAM_CHUNK = 1ull << 22;   // rays per pipelined chunk of the host-buffer entry points
constexpr int TAIL_RING = 4;                     // tail queues shared round robin by ray-stream launches (see trace_device)
constexpr int64_t COOP_MAX_LIMIT = 16;           // upper bound of B2RT_OPT_COOP_MAX: the tail queues hold this many records per warp
constexpr uint64_t NEXT_RING = 256;             // per-launch ray counters of the persistent kernels (b2rt_context::d_next)

extern std::string g_create_error;
struct Group;
struct Comm;

}  // namespace b2rt_detail

using b2rt_detail::Buffer;

struct ModeTrial { int calls = 0; float ms[2] = { 0.0f, 0.0f }; int choice = -1; };

struct b2rt_context {
    int device = 0;
    int sm_count = 0;
    size_t l2_persist_max = 0, l2_window_max = 0;   // cudaDeviceProp persistingL2CacheMaxSize / accessPolicyMaxWindowSize
    cudaStream_t stream = nullptr, stream_in = nullptr, stream_out = nullptr;
    std::unordered_map<uint64_t, Buffer> buffers;
    uint64_t next_id = 1;
    b2rt_buffer bound[4] = { 0, 0, 0, 0 };
    bool arg_set[B2RT_ARG_COUNT] = { false };
    uint32_t width = 0, height = 0, frame_count = 0, frame_seed = 0;
    int32_t bounces = 0, light_type = 0;
    float sky = 0.0f;
    float cam_pos[4] = { 0, 0, 0, 0 }, cam_front[4] = { 0, 0, 0, 0 }, cam_up[4] = { 0, 0, 0, 0 };
    // derived scene
    bool scene_dirty = true;
    void *d_wide = nullptr, *d_leaf = nullptr, *d_shade = nullptr;      // d_leaf points into d_wide's allocation (alloc_bvh)
    size_t bvh_bytes = 0, l2_window_bytes = 0;
    uint32_t *d_child_bin = nullptr, *d_leaf_dir = nullptr;   // refit support: binary node behind every wide child slot / leaf block
    b2rt_scene_info info;
    uint32_t stack_bound = 8;
    b2rt::SceneView view;
    // scratch
    unsigned long long* d_next = nullptr;      // NEXT_RING counter blocks (4 x u64: ray counter, tail-queue length, tail-queue read
    uint64_t next_seq = 0;                     // position, pad), one per in-flight ray-stream launch
    // cooperative tail mode: queues of unfinished rays, one per launch that may be in flight at the same time
    void* d_tail[b2rt_detail::TAIL_RING + 4] = { nullptr };  // [0, TAIL_RING): ray-stream launches (one per stream in use); then one per wavefront lane
    bool tail_two_step[b2rt_detail::TAIL_RING + 4] = { false };   // the slot was allocated with the second queue of the two-step tail
    unsigned long long tail_slot_stream[b2rt_detail::TAIL_RING] = { 0 };   // stream id + 1 that owns ray-stream slot i (0 = free) ...
    uint64_t tail_slot_used[b2rt_detail::TAIL_RING] = { 0 };               // ... and the launch number of its last use
    uint64_t tail_capacity_records = 0;
    uint32_t tail_rec_words = 0;
    int grid_tail = 0;
    unsigned long long* d_counters = nullptr;
    void* d_stage_rays[2] = { nullptr, nullptr };
    void* d_stage_out[2] = { nullptr, nullptr };
    uint64_t stage_capacity = 0;               // rays per staging buffer ...
    size_t stage_out_bytes = 0;                // ... and bytes per output staging buffer
    void* d_stage_in2[2] = { nullptr, nullptr };   // second input of a host-buffer entry (b2rt_trace_radiance: the seeds) ...
    size_t stage_in2_bytes = 0;                // ... and its bytes per staging buffer
    // wavefront frame path: two ray queues, hits, per-path state, three rotating queue counters
    void* d_wf_rays[2] = { nullptr, nullptr };
    void *d_wf_hits = nullptr, *d_wf_state = nullptr;
    unsigned long long* d_wf_count = nullptr;
    uint64_t wf_capacity = 0;
    cudaStream_t wf_stream[4] = { nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t ev_wf_fork = nullptr, ev_wf_join[4] = { nullptr, nullptr, nullptr, nullptr };
    std::map<std::pair<uint64_t, int>, ModeTrial> tuner;   // render-mode auto-tuning per launch shape (work items, bounces)
    std::pair<uint64_t, int> tune_pending_key;
    int tune_pending_mode = -1;
    cudaEvent_t ev_tune[2] = { nullptr, nullptr };
    cudaEvent_t ev_refit[2] = { nullptr, nullptr };   // b2rt_refit_scene_device, b2rt_trace_radiance_device: caller's stream -> context's stream and back
    void* d_rgba8 = nullptr;            // 8-bit read-back staging
    uint64_t rgba8_capacity = 0;
    cudaEvent_t ev_in[2] = { nullptr, nullptr }, ev_comp[2] = { nullptr, nullptr }, ev_out[2] = { nullptr, nullptr };
    // options
    int64_t opt_traversal = 0, opt_counters = 0, opt_blocks_per_sm = 0, opt_render_mode = 2, opt_refill_min = 6, opt_leaf_bias = 0, opt_wf_lanes = 0, opt_coop_max = -1, opt_l2_persist = 1, opt_stage_times = 0, opt_wf_grid_split = 0, opt_resume_max = 0, opt_tail_help = 1, opt_shard_fence = 1;
    uint32_t tail_tag_seq = 0;                 // tag of the last persistent launch's tail records (kernels.h)
    int grid_closest = 0, grid_any = 0;
    uint64_t launches = 0;
    // stage timing of the wavefront frame path (B2RT_OPT_STAGE_TIMES): events recorded around the stages of wavefront 0
    std::vector<cudaEvent_t> stage_events;
    std::vector<uint32_t> stage_kinds;       // kind of the stage that ENDS at event i + 1
    uint32_t stage_used = 0;
    // ---- multi-GPU (multi.cu) ----
    b2rt_detail::Group* group = nullptr;     // this handle drives several devices of this process (b2rt_create_multi)
    b2rt_context* parent = nullptr;          // this context is a member of parent's group
    b2rt_detail::Comm* comm = nullptr;       // this handle is one rank of a multi-process job (b2rt_comm_init)
    float* mirror = nullptr;                 // frame path: finished pixels are also stored here (the root's image, peer-mapped)
    void* mirror_ipc_base = nullptr;         // ... opened from another process with cudaIpcOpenMemHandle
    std::string error;
};


namespace b2rt_detail {

int fail(b2rt_context* c, int status, const std::string& msg);
int cuda_fail(b2rt_context* c, cudaError_t e, const char* what);
int use_device(b2rt_context* ctx);
Buffer* find(b2rt_context* ctx, b2rt_buffer id);
int ensure_scene(b2rt_context* ctx);
void free_scene(b2rt_context* ctx);
int alloc_bvh(b2rt_context* ctx, size_t wide_bytes, size_t leaf_bytes);   // one allocation for wide nodes + leaf blocks
void free_tail(b2rt_context* ctx);
void scene_l2_setup(b2rt_context* ctx);
int buffer_create_single(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out, bool zero_fill);
bool context_alive(const b2rt_context* ctx);

// What install_scene needs to know about a freshly derived compressed wide BVH (host: wide_bvh.cpp, device: scene_build.cu).
struct DerivedScene {
    uint64_t n_tris, n_nodes, n_wide_nodes, n_leaf_blocks;
    size_t wide_bytes, leaf_bytes, shade_bytes;
    uint32_t max_depth_binary, max_depth_wide, stack_bound;
};
// The derived arrays are in place (d_wide / d_leaf / d_shade / d_child_bin / d_leaf_dir): scene info, SceneView, launch
// geometry, L2 set-up and tail queues for them; the peers of a device group take copies. Clears scene_dirty.
int install_scene(b2rt_context* ctx, const DerivedScene& d);
// refit.cu: per-triangle shading records (normals + material) of `tris`
cudaError_t launch_shade_records(b2rt::ShadeTri* shade, const b2rt::RefTriangle* tris, uint32_t n, cudaStream_t s);
int render_items(b2rt_context* ctx, const b2rt::GidMap& map, uint64_t n);
// `to` waits for the work enqueued on `from` so far (ev: one of the context's events; the wait takes the recorded state, so
// the event can be recorded again by the next call).
cudaError_t stream_edge(cudaEvent_t ev, cudaStream_t from, cudaStream_t to);

// multi.cu
void group_destroy(b2rt_context* ctx);
void comm_destroy(b2rt_context* ctx);
int group_buffer_create(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out);
int group_each(b2rt_context* ctx, int (*fn)(b2rt_context*, void*), void* arg, bool parallel);
int group_adopt_scene(b2rt_context* root);
int group_execute(b2rt_context* ctx, size_t gid_begin, size_t gid_end);
// Items [0, n) of a host-buffer entry: member k runs fn(member, first, count) over its contiguous range [n*k/world,
// n*(k+1)/world); empty ranges are skipped.
int group_split(b2rt_context* ctx, uint64_t n, const std::function<int(b2rt_context*, uint64_t, uint64_t)>& fn);
int group_finish(b2rt_context* ctx);
void group_bind_output(b2rt_context* ctx);
int group_broadcast_buffer(b2rt_context* ctx, b2rt_buffer id);   // the root's contents of buffer `id` to every peer's copy
const std::vector<b2rt_context*>& group_members(const b2rt_context* ctx);

}  // namespace b2rt_detail

#define CK(call)                                                                     \
    do {                                                                             \
        cudaError_t e__ = (call);                                                    \
        if (e__ != cudaSuccess) return b2rt_detail::cuda_fail(ctx, e__, #call);      \
    } while (0)
