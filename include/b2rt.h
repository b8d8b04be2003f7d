/* b2rt.h -- C ABI of libb2rt.so: the B200 (sm_100a) replacement for the device
 * side of Mini-OpenCL-Raytracer, i.e. everything the reference reaches through
 * its OpenCL wrapper layer CLutils.{h,cpp} (CLContext / CLKernel, the drop-in
 * boundary of SURVEY.md 8b) plus a ray-stream entry the reference lacks.
 *
 * Plain C: opaque handle, plain pointers and sizes, int status returns, no
 * exceptions and no torch/CUDA types in any signature. One host thread per
 * handle at a time. There is NO CPU fallback: every entry point fails with
 * B2RT_DEVICE_NOT_FOUND when no CUDA device is usable.
 *
 * Citations are file:line in the reference tree (/root/reference).
 */
#ifndef B2RT_H
#define B2RT_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2RT_VERSION 100

/* Status codes reuse the OpenCL numbering so that the host wrappers can turn
 * them into the same CLException text as the reference (CLutils.h:29-114). */
enum {
    B2RT_SUCCESS = 0,
    B2RT_DEVICE_NOT_FOUND = -1,             /* CL_DEVICE_NOT_FOUND */
    B2RT_MEM_OBJECT_ALLOCATION_FAILURE = -4,
    B2RT_OUT_OF_RESOURCES = -5,             /* any CUDA runtime failure */
    B2RT_OUT_OF_HOST_MEMORY = -6,
    B2RT_INVALID_VALUE = -30,
    B2RT_INVALID_CONTEXT = -34,
    B2RT_INVALID_MEM_OBJECT = -38,
    B2RT_INVALID_ARG_INDEX = -49,
    B2RT_INVALID_ARG_VALUE = -50,
    B2RT_INVALID_ARG_SIZE = -51,
    B2RT_INVALID_KERNEL_ARGS = -52,
    B2RT_INVALID_GLOBAL_WORK_SIZE = -63
};

/* The 14 argument slots of KernelEntry (kernel_bvh.cl:415-431), numbered like
 * RenderKernelArgument_t (CLutils.h:11-27). */
enum {
    B2RT_ARG_BUFFER_OUT = 0,       /* b2rt_buffer: W*H*16 B accumulation image     */
    B2RT_ARG_BUFFER_SCENE = 1,     /* b2rt_buffer: CLTriangle[]  (256 B each)      */
    B2RT_ARG_BUFFER_NODE = 2,      /* b2rt_buffer: CLLinearBVHNode[] (48 B each)   */
    B2RT_ARG_BUFFER_MATERIAL = 3,  /* b2rt_buffer: CLMaterial[]  (64 B each)       */
    B2RT_ARG_WIDTH = 4,            /* uint32 */
    B2RT_ARG_HEIGHT = 5,           /* uint32 */
    B2RT_ARG_FRAME_COUNT = 6,      /* uint32 */
    B2RT_ARG_FRAME_SEED = 7,       /* uint32, accepted and ignored like the kernel does */
    B2RT_ARG_LIGHT_BOUNCES = 8,    /* int32  */
    B2RT_ARG_LIGHT_TYPE = 9,       /* int32  */
    B2RT_ARG_SKYBOX_INTENSITY = 10,/* float  */
    B2RT_ARG_CAMERA_POS = 11,      /* 16-byte float3 (CLRaytracer.cpp:42-47 passes sizeof(float3)) */
    B2RT_ARG_CAMERA_FRONT = 12,
    B2RT_ARG_CAMERA_UP = 13,
    B2RT_ARG_COUNT = 14
};

/* cl_mem_flags subset used by the reference (CLBVHnode.cpp:215, CLRaytracer.cpp:133). */
enum {
    B2RT_MEM_WRITE_ONLY = 1 << 1,
    B2RT_MEM_READ_ONLY = 1 << 2,
    B2RT_MEM_COPY_HOST_PTR = 1 << 5
};

typedef struct b2rt_context b2rt_context;   /* replaces CLContext + CLKernel (CLutils.h:116-145) */
typedef uint64_t b2rt_buffer;               /* replaces cl::Buffer; 0 is never a valid buffer */

/* Ray-stream records (new API; the reference only traces camera paths inside
 * its megakernel). dir need not be unit length: it is normalised exactly like
 * InitRay (kernel_bvh.cl:42-55). tmin is accepted for layout compatibility and
 * IGNORED, because the reference's RayTriangle has no lower bound on t
 * (kernel_bvh.cl:140); tmax seeds isect.t (the reference uses 100000). */
typedef struct { float ox, oy, oz, tmin; float dx, dy, dz, tmax; } b2rt_ray;   /* 32 B */
typedef struct { float t, u, v; uint32_t tri; } b2rt_hit;                       /* 16 B */
#define B2RT_MISS 0xFFFFFFFFu
#define B2RT_MAX_RENDER_DIST 100000.0f      /* kernel_bvh.cl:7 */

typedef struct {
    uint64_t n_triangles, n_nodes, n_materials;      /* reference-layout inputs           */
    uint64_t n_wide_nodes, n_leaf_blocks;             /* GPU-resident compressed wide BVH  */
    uint64_t wide_node_bytes, leaf_bytes, shading_bytes;
    uint32_t max_depth_binary, max_depth_wide;
    uint32_t sm_count, reserved;
} b2rt_scene_info;

typedef struct {
    uint64_t rays;              /* rays traced by counted launches                         */
    uint64_t wide_nodes;        /* wide-node visits                                        */
    uint64_t leaf_blocks;       /* leaf blocks fetched                                     */
    uint64_t leaf_gate_pass;    /* ... of which passed the exact fp32 leaf box             */
    uint64_t tri_tests;         /* Moller-Trumbore evaluations                             */
    uint64_t bytes_fetched;     /* algorithmic (requested) bytes: 84 B per wide-node visit (5 x 16 B + one 4-byte order word of
                                   the 112-byte record) + 48 B per record of every leaf block fetched (+ 32 B for the few blocks
                                   that carry an explicit box) */
    /* warp scheduling of the persistent kernels: phases run and lanes that took part in them */
    uint64_t node_phases, node_phase_lanes, leaf_phases, leaf_phase_lanes, refills, refill_lanes;
    uint64_t max_steps_per_ray; /* node + leaf steps of the most expensive ray (tail detector; solo steps only) */
    uint64_t stack_overflows;   /* lanes whose traversal stack (counting build) or cooperative frontier (every build) overflowed:
                                   always 0 for trees that passed upload validation, whose exact bound sizes the stack      */
    uint64_t coop_rays;         /* rays finished by the warp-cooperative tail mode ...                                   */
    uint64_t coop_steps;        /* ... and the node + leaf visits done for them                                          */
    uint64_t coop_max_steps;    /* node + leaf visits of the most expensive ray of the cooperative tail mode ...         */
    uint64_t coop_max_rounds;   /* ... and the most rounds (memory round trips) one ray took there                       */
    uint64_t resumed_rays;      /* suspended rays picked up again by the second persistent pass of the two-step tail     */
} b2rt_counters;

enum {
    B2RT_OPT_TRAVERSAL = 0,     /* 0 = compressed wide BVH (default), 1 = reference-layout binary walk */
    B2RT_OPT_COUNTERS = 1,      /* 1 = launches use the counting build of the kernels      */
    B2RT_OPT_BLOCKS_PER_SM = 2, /* persistent grid = value * SM count (0 = default)        */
    B2RT_OPT_RENDER_MODE = 3,   /* frame path: 0 = wavefront (generate, then trace + shade/compact per bounce), 1 = megakernel
                                   (one thread per pixel, like KernelEntry), 2 = whichever of the two measures faster for the
                                   launch shape at hand (default). Frames are bit-identical in every mode. */
    B2RT_OPT_REFILL_MIN = 4,    /* idle lanes of a warp that trigger a ray refill (1..32, default 6) */
    B2RT_OPT_LEAF_BIAS = 5,     /* weight of the leaf vote in sixteenths (16 = plain majority; 0 = default: 32 closest-hit and frames, 48 any-hit) */
    B2RT_OPT_WAVEFRONT_LANES = 6, /* wavefront frame path: independent wavefronts in flight per launch, 1..4 (0 = by size) */
    B2RT_OPT_L2_PERSIST = 8,    /* 1 (default): the wide-node array is kept resident in L2 by an access-policy window (persisting
                                   carve-out sized to it) on every stream that runs traversal kernels; 0 = plain caching.
                                   Results do not depend on it. */
    B2RT_OPT_STAGE_TIMES = 9,   /* 1: the wavefront frame path records a CUDA event after every stage of the launch's first wavefront;
                                   read the durations with b2rt_stage_times (profiling aid, default 0) */
    B2RT_OPT_WAVEFRONT_GRID_SPLIT = 10, /* wavefront frame path with several wavefronts in flight: 1 = each one's persistent grids take an
                                   equal part of the device's CTA slots, so that one wavefront's latency-bound stage tails run next to
                                   another's bulk traversal instead of queueing behind a full-device grid; 0 = every grid sized for the
                                   whole device. Results do not depend on it. */
    B2RT_OPT_RESUME_MAX = 11,   /* two-step tail: a dry warp with at most this many live rays suspends them; a second persistent launch
                                   re-packs all suspended rays 32 to a warp and walks on at full width, and only what that pass
                                   leaves (B2RT_OPT_COOP_MAX per warp) goes to the cooperative kernel. 0 = off (default, also -1) .. 16.
                                   Only used while larger than the cooperative threshold. Results do not depend on it. Ignored by
                                   b2rt_trace_multi[_device]. */
    B2RT_OPT_TAIL_HELP = 12,    /* 1 (default) / 0: in a library built with -DB2_TAIL_HELP=1, warps of a persistent traversal launch that have
                                   finished or handed over their own rays serve the cooperative tail queue inside the same launch; the
                                   tail kernel takes what is left. The default build compiles this out (measured slower on frame shares,
                                   DESIGN.md 4c), the option is then accepted and ignored. Results do not depend on it. */
    B2RT_OPT_SHARD_FENCE = 13,  /* 1 (default) / 0: b2rt_execute_shard with a mapped root image starts with a 4-byte ncclAllReduce, so that no
                                   rank's kernels store pixels of the new frame into rank 0's image while rank 0 is still reading the
                                   previous one (b2rt_read_pixels is asynchronous). A job that never reads between two frames may set 0 on
                                   EVERY rank (the fence is a collective). Results do not depend on it. */
    B2RT_OPT_COOP_MAX = 7       /* tail mode of the persistent kernels: a warp whose ray pool is dry and that has at most this many
                                   rays alive hands them to the cooperative tail kernel, 32 lanes per ray (0 = off .. 16; default -1 = 8, but off for scenes
                                   of fewer than ~1000 nodes, whose rays are too short to gain). Results do not
                                   depend on it. Ignored by b2rt_trace_multi[_device], whose launches have no cooperative tail. */
};

/* ---- lifetime ---------------------------------------------------------------------- */
/* CLContext::CLContext + CLKernel::CLKernel (CLutils.cpp:9-35, 52-66): pick the
 * device, create the stream (the in-order queue), load the precompiled kernels. */
int b2rt_create(int device_id, b2rt_context** out);
void b2rt_destroy(b2rt_context* ctx);
/* Text of the last failure on this context (or of the last failed b2rt_create when ctx == NULL). */
const char* b2rt_last_error(const b2rt_context* ctx);
const char* b2rt_status_string(int status);          /* GetClErrorString (CLutils.h:29-105) */

/* ---- buffers and kernel arguments ----------------------------------------------------- */
/* cl::Buffer(context, flags, size, host_ptr, &err) (CLBVHnode.cpp:214-235,
 * CLRaytracer.cpp:132-135). With COPY_HOST_PTR the bytes are copied before return.
 * Buffers without host data are zero-filled: the reference never clears its
 * accumulation buffer although frame 1 reads it (kernel_bvh.cl:454). */
int b2rt_buffer_create(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out);
int b2rt_buffer_release(b2rt_context* ctx, b2rt_buffer buf);
/* clSetKernelArg as used by CLKernel::SetArgument (CLutils.cpp:68-77). Slots 0-3
 * take a pointer to a b2rt_buffer (size 8), the others the scalar / float3 sizes above. */
int b2rt_set_arg(b2rt_context* ctx, uint32_t slot, const void* data, size_t size);

/* ---- frame path: CLContext::ExecuteKernel / ReadBuffer / Finish (CLutils.cpp:37-50) ---- */
/* Enqueue KernelEntry for gid in [0, global_work_size). Asynchronous. */
int b2rt_execute(b2rt_context* ctx, size_t global_work_size);
/* Same, restricted to gid in [gid_begin, gid_end): one screen shard of a multi-GPU frame. */
int b2rt_execute_range(b2rt_context* ctx, size_t gid_begin, size_t gid_end);
/* Same, for n_bands bands of band_pixels consecutive gids whose starts are stride_pixels apart, beginning at
 * gid_begin: everything one rank of a multi-GPU frame draws (e.g. every world-th 8-row band), as ONE launch
 * sequence instead of one per band. */
int b2rt_execute_bands(b2rt_context* ctx, size_t gid_begin, uint32_t band_pixels, uint32_t stride_pixels, uint32_t n_bands);
/* Non-blocking read of `bytes` from offset 0 of `buf` into host memory (CLutils.cpp:37-42). */
int b2rt_read_buffer(b2rt_context* ctx, b2rt_buffer buf, void* dst, size_t bytes);
int b2rt_finish(b2rt_context* ctx);
/* Optional: page-lock a host range that b2rt_read_buffer / the ray-stream calls will be given repeatedly
 * (e.g. CLRaytracer::pixels, CLRaytracer.cpp:127), so that the copies run at full PCIe speed and truly
 * asynchronously. The reference's OpenCL runtime pins its staging memory itself; here it is explicit. */
int b2rt_host_register(b2rt_context* ctx, void* ptr, size_t bytes);
int b2rt_host_unregister(b2rt_context* ctx, void* ptr);

/* ---- convenience wrappers over the calls above --------------------------------------- */
/* CLBVHScene::SetupBuffers (CLBVHnode.cpp:209-236): three buffer creates + binds. */
int b2rt_upload_scene(b2rt_context* ctx, const void* triangles, uint64_t n_triangles,
                      const void* nodes, uint64_t n_nodes, const void* materials, uint64_t n_materials);
/* CLRaytracer::SetupBuffers (CLRaytracer.cpp:122-137): WIDTH/HEIGHT + zeroed output buffer. */
int b2rt_resize(b2rt_context* ctx, uint32_t width, uint32_t height);
int b2rt_read_pixels(b2rt_context* ctx, void* dst, size_t bytes);   /* read_buffer on the bound slot 0 */
/* Display read-back: the first bytes/4 pixels of the bound output image clamped to [0,1] and quantised to 8-bit
 * RGBA (alpha 255) on the device, then copied (non-blocking, finish with b2rt_finish). 4 B/pixel over PCIe instead
 * of the 16 B/pixel the reference reads back and hands to glTexImage2D(GL_RGBA, GL_FLOAT) (CLRaytracer.cpp:55,64-67).
 * The accumulation image itself is not modified. */
int b2rt_read_pixels_rgba8(b2rt_context* ctx, void* dst, size_t bytes);

/* ---- BVH build on the device (new) ------------------------------------------------------ */
/* Stands in for CLBVHScene::RecursiveBuild + FlattenBVHTree (CLBVHnode.cpp:7-183): builds a binary BVH over
 * `triangles` (CLTriangle[n] in LOADER order, host memory) on the GPU -- Morton order, Karras hierarchy, bottom-up
 * boxes -- and returns it in the reference's own format: nodes_out receives CLLinearBVHNode[*n_nodes_out] (pre-order,
 * first child at index+1, at most 2n-1 nodes), order_out[k] the input index of the triangle that must become triangle
 * k of the scene array (the caller re-orders its triangles like CreateBVHTrees does, CLBVHnode.cpp:197). The tree is
 * NOT the reference's SAH tree: hit IDs refer to this order, and where the reference's result depends on visiting
 * order (equal-t ties, negative t) the winner can differ from a scene built by the host builder. */
int b2rt_build_bvh(b2rt_context* ctx, const void* triangles, uint64_t n_triangles, void* nodes_out, uint64_t nodes_capacity,
                   uint64_t* n_nodes_out, uint32_t* order_out);

/* Scene build on the device (new). d_triangles = CLTriangle[n_triangles] in LOADER order in device memory of this
 * handle's device (the root device of a group; device or managed memory, else B2RT_INVALID_VALUE). Builds the binary BVH
 * exactly like b2rt_build_bvh does from the same triangles (same groups, byte-identical nodes and order), re-orders the
 * triangles on the device, creates two new buffers -- the re-ordered CLTriangle[] and the CLLinearBVHNode[] -- binds them
 * to slots 1 and 2 (previously bound buffers are unbound, not released) and derives the compressed wide BVH on the device,
 * byte-identical to what b2rt_upload_scene derives on the host from the same arrays: no host copy of the scene is made.
 * On a b2rt_create_multi handle the root builds and every device gets copies. Bind the material buffer (slot 3) first.
 * d_order_out (may be NULL): device uint32[n_triangles], order[k] = input index of triangle k. Rejects a NULL or empty
 * array, n_triangles >= 2^31 - 1 (B2RT_INVALID_VALUE) and non-finite vertex positions or unquantisable bounds
 * (B2RT_INVALID_ARG_VALUE); after a failure the previously bound scene is still usable. Rebinding slot 1, 2 or 3 later
 * falls back to the host derivation; b2rt_refit_scene works on the device-built scene. The build is ordered behind the
 * work already enqueued on cuda_stream (NULL = the context's stream) and is synchronous on return. */
int b2rt_build_scene_device(b2rt_context* ctx, const void* d_triangles, uint64_t n_triangles, uint32_t* d_order_out,
                            b2rt_buffer* triangles_out, b2rt_buffer* nodes_out, uint64_t* n_nodes_out, void* cuda_stream);

/* Refit (new): `triangles` = CLTriangle[n_triangles] with NEW vertex data for the bound scene, same count and order
 * (animated / deformed geometry). The bound triangle buffer is replaced, the bound CLLinearBVHNode buffer gets the boxes
 * refitted bottom-up (read it back with b2rt_read_buffer to see the tree in the reference's format), and the compressed
 * wide BVH -- quantised child boxes, leaf blocks, shading records -- is refreshed in place by device kernels; topology,
 * triangle order and therefore hit IDs stay. Stands in for re-running CLBVHScene::RecursiveBuild (CLBVHnode.cpp:7-159) +
 * SetupBuffers for every frame of an animation. Results equal the reference's walk over (new triangles, refitted nodes).
 * Fails (rebuild instead) when two triangles that were the loader's copies of one face no longer are. Synchronous. */
int b2rt_refit_scene(b2rt_context* ctx, const void* triangles, uint64_t n_triangles);

/* Refit from device memory (new): the same contract as b2rt_refit_scene (same topology, order and hit IDs; results equal
 * the reference's walk over the new triangles and the refitted nodes), but the new vertex data is already on this
 * handle's device and nothing crosses PCIe -- e.g. the animation loop "simulate (torch) -> refit -> trace / render" on one
 * stream without a host round trip.
 *  d_triangles: CLTriangle records, 16-byte aligned, device or managed memory of the handle's (root) device.
 *  d_order == NULL: d_triangles holds the n scene-order triangles. It may be the bound triangle buffer itself (in place).
 *  d_order != NULL: device uint32[n]; scene triangle k is d_triangles[d_order[k]]. This is exactly the d_order_out of
 *                   b2rt_build_scene_device (or b2rt_build_bvh's order_out), so loader-order data can be passed as is.
 *  d_status: device uint32, required. The call sets it to 0 on the stream, then ORs in B2RT_REFIT_* bits.
 *  Ordered after the work already enqueued on cuda_stream (NULL = the context's stream) and on the context's stream
 *  (which frames in flight on the wavefront path join). Work enqueued after the call on either stream sees the refitted
 *  scene; work on any third stream is the caller's to order. On a single-device handle the call returns without waiting
 *  for the device (only the first call after binding a new scene derives it, which waits). On a b2rt_create_multi handle
 *  the root gathers, the peers receive copies and every device refits its own; the call is synchronous there and d_status
 *  holds the OR of every device's bits when it returns.
 * Returns B2RT_INVALID_CONTEXT for a NULL handle, B2RT_INVALID_KERNEL_ARGS when no built scene is bound, B2RT_INVALID_VALUE
 * for a NULL or empty input or a NULL d_status, n_triangles different from the bound scene's count, a pointer that is not
 * device or managed memory of the right device, d_triangles not 16-byte or d_order / d_status not 4-byte aligned, and
 * d_triangles overlapping the bound triangle buffer when d_order is given (a gather cannot run in place) or overlapping it
 * without being exactly it. Nothing of the scene is touched before these checks pass.
 * A non-zero status leaves a scene that is safe to traverse but whose hits are undefined: topology and all indices are
 * unchanged, only positions and boxes are stale or wrong. A later refit with valid data restores the scene completely,
 * because a refit is a pure function of (topology, triangles). */
int b2rt_refit_scene_device(b2rt_context* ctx, const void* d_triangles, uint64_t n_triangles, const uint32_t* d_order,
                            uint32_t* d_status, void* cuda_stream);
/* Status bits of b2rt_refit_scene_device. b2rt_refit_scene reports these conditions as B2RT_INVALID_ARG_VALUE, except that
 * it checks vertices for non-finite values only through the boxes they produce. */
enum {
    B2RT_REFIT_NONFINITE = 1,      /* a non-finite vertex coordinate (every vertex is checked)                       */
    B2RT_REFIT_DUPLICATE = 2,      /* two triangles that were the loader's copies of one face no longer are: rebuild */
    B2RT_REFIT_RANGE = 4,          /* bounds too large to quantise                                                   */
    B2RT_REFIT_LEAF_BOX = 8,       /* a leaf block without a stored box no longer matches its vertices               */
    B2RT_REFIT_ORDER = 16          /* some d_order[k] >= n: scene triangle k was left as it was                      */
};

/* ---- ray-stream path (new) ----------------------------------------------------------- */
/* Host buffers: H2D copy, trace, D2H copy, synchronous on return.
 * closest: hits[i] = {t,u,v,tri} of Intersect() (kernel_bvh.cl:171-219), tri = B2RT_MISS and
 * t = tmax on a miss. any: occluded[i] = Intersect(tmax).hit with early exit. */
int b2rt_trace_closest(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, b2rt_hit* hits);
int b2rt_trace_any(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, uint32_t* occluded);
/* Device-resident buffers (plain device pointers, e.g. torch tensor data_ptr()); enqueued on
 * `cuda_stream` (a cudaStream_t passed as void*; NULL = the context's own stream). Asynchronous.
 * Every launch has its own work counter, so launches on different streams may overlap; on at most 4
 * DIFFERENT streams at a time while the cooperative tail mode is on (B2RT_OPT_COOP_MAX > 0): a tail queue belongs to
 * the stream whose launches use it (allocated by that stream's first launch), and a fifth stream takes over the
 * queue of the stream that has not launched for longest. */
int b2rt_trace_closest_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, b2rt_hit* d_hits, void* cuda_stream);
int b2rt_trace_any_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, uint32_t* d_occluded, void* cuda_stream);

/* The k nearest hits per ray (new). Intersect() (kernel_bvh.cl:171-219) with isect replaced by a list of at most k hits:
 *  - the walk is the reference's depth-first order; a leaf is entered iff its exact fp32 box passes RayBounds on
 *    [0, bound], where bound = tmax while the list holds fewer than k hits and the t of its k-th entry once it is full;
 *  - a triangle is accepted iff RayTriangle accepts it with t < bound: the acceptance rule of b2rt_trace_closest (no lower
 *    bound on t, tmin ignored, front faces only). The bound is updated after every insertion, also between the triangles
 *    of one leaf;
 *  - an accepted hit is inserted after every entry with t <= its own (equal t keeps visiting order, like the reference's
 *    strict <); a full list drops its last entry;
 *  - the ray ends when bound < 0 (no later box can pass);
 *  - row i of the output is hits[i*k .. i*k+k), sorted by t; unused slots are {t = tmax, u = 0, v = 0, tri = B2RT_MISS}.
 * Every triangle of the scene array is its own hit: the loader's two copies of a face (SURVEY.md A-6) appear as two hits,
 * usually at the same t. With k = 1 every row is bit-identical to what b2rt_trace_closest returns, misses included.
 * k = 0 or k > B2RT_MULTI_MAX_HITS, or a NULL pointer with n > 0, returns B2RT_INVALID_VALUE and writes nothing; n = 0
 * succeeds and does nothing.
 * b2rt_trace_multi: host buffers, synchronous (pipelined in chunks like b2rt_trace_closest; a chunk holds fewer rays for
 * larger k). On a b2rt_create_multi handle the rays are cut into contiguous ranges, one per device.
 * b2rt_trace_multi_device: device buffers (d_hits = b2rt_hit[n * k]), asynchronous on cuda_stream with the stream rules of
 * b2rt_trace_closest_device; on a b2rt_create_multi handle it runs on the root.
 * B2RT_OPT_TRAVERSAL = 1 runs the query through the reference-layout walk, B2RT_OPT_COUNTERS = 1 through the counting
 * build. These launches have no cooperative tail: B2RT_OPT_COOP_MAX and B2RT_OPT_RESUME_MAX are accepted and ignored. */
#define B2RT_MULTI_MAX_HITS 64
int b2rt_trace_multi(b2rt_context* ctx, const b2rt_ray* rays, uint64_t n, uint32_t k, b2rt_hit* hits);
int b2rt_trace_multi_device(b2rt_context* ctx, const b2rt_ray* d_rays, uint64_t n, uint32_t k, b2rt_hit* d_hits, void* cuda_stream);

/* ---- closest point (new) ------------------------------------------------------------------ */
/* Nearest surface point of the bound scene to each query point, and its squared distance (collision and contact, snapping
 * onto a surface, distance-field sampling, attribute transfer).
 *  Candidates: every triangle k of the bound scene array, (a, b, c) = (v1, v2, v3).position.xyz of its CLTriangle. The
 *    loader's two copies of a face are two candidates (the second one's vertices rotated as stored).
 *  Distance: cp(p, a, b, c) -> (d2, u, v) is Ericson's region test ("Real-Time Collision Detection" 5.1.5), every operation
 *    one IEEE fp32 operation rounded to nearest, no contraction, in this order: ab = b-a, ac = c-a, ap = p-a, d1 = ab.ap,
 *    d2' = ac.ap (x.y = (x0*y0 + x1*y1) + x2*y2); bp = p-b, cp = p-c, d3 = ab.bp, d4 = ac.bp, d5 = ab.cp, d6 = ac.cp,
 *    vc = d1*d4 - d3*d2', vb = d5*d2' - d1*d6, va = d3*d6 - d5*d4. The first region (Ericson's order and conditions) that
 *    holds is taken (an edge region also needs its denominator > 0, which only a zero-length edge fails: without it a
 *    repeated vertex would take that edge's branch with t = 0/0):
 *      vertex a   d1 <= 0 && d2' <= 0                         (u, v) = (0, 0), point a
 *      vertex b   d3 >= 0 && d4 <= d3                         (1, 0), point b
 *      edge ab    vc <= 0 && d1 >= 0 && d3 <= 0 && d1-d3 > 0                      (t, 0), t = d1/(d1-d3), point a + ab*t
 *      vertex c   d6 >= 0 && d5 <= d6                                              (0, 1), point c
 *      edge ac    vb <= 0 && d2' >= 0 && d6 <= 0 && d2'-d6 > 0                    (0, t), t = d2'/(d2'-d6), point a + ac*t
 *      edge bc    va <= 0 && (d4-d3) >= 0 && (d5-d6) >= 0 && (d4-d3)+(d5-d6) > 0
 *                                                                (1-t, t), t = (d4-d3)/((d4-d3)+(d5-d6)), point b + (c-b)*t
 *      interior   (va+vb)+vc > 0: denom = 1/((va+vb)+vc), (u, v) = (vb*denom, vc*denom), point (a + ab*u) + ac*v
 *      otherwise (degenerate): the edges ab, ac, bc in this order from their origins a, a, b, each with
 *        t = clamp01((o->p).e / e.e) (clamp01 maps NaN to 0), point o + e*t, clamped and measured as below; the smallest
 *        d2 wins, ties to the earlier edge; (u, v) = (t, 0), (0, t) or (1-t, t).
 *    The point is clamped per axis into the triangle's vertex box [min(a,b,c), max(a,b,c)] (fminf(fmaxf(q, lo), hi): NaN
 *    becomes lo), then d2 = ((px-qx)^2 + (py-qy)^2) + (pz-qz)^2. (u, v) are the branch's parameters in the reference's
 *    barycentric convention, point = (1-u-v) v1 + u v2 + v v3.
 *  Result: among the candidates with d2 <= max_d2, the smallest d2, ties to the smallest triangle index:
 *    out[i] = {d2, u, v, tri}; when none qualifies {max_d2, 0, 0, B2RT_MISS}. max_d2 = +inf searches the whole scene; a
 *    negative or NaN max_d2, or a NaN coordinate, always misses. The result does not depend on the tree or visiting order.
 *  Outside the contract: scenes with non-finite vertices (the device build and refit reject them) and caller-supplied trees
 *    whose node boxes do not contain their triangles (every builder here produces boxes that do).
 * n = 0 succeeds; a NULL pointer with n > 0 returns B2RT_INVALID_VALUE and writes nothing.
 * b2rt_closest_point: host buffers, synchronous, pipelined in chunks like b2rt_trace_closest; on a b2rt_create_multi handle
 * the queries are cut into contiguous ranges, one per device.
 * b2rt_closest_point_device: device buffers, asynchronous on cuda_stream with the stream rules of b2rt_trace_closest_device;
 * on a b2rt_create_multi handle it runs on the root.
 * B2RT_OPT_TRAVERSAL = 1 runs the reference-layout walk, B2RT_OPT_COUNTERS = 1 the counting build (rays = queries,
 * tri_tests = distance evaluations). B2RT_OPT_COOP_MAX, B2RT_OPT_RESUME_MAX and B2RT_OPT_TAIL_HELP are ignored. */
typedef struct { float x, y, z, max_d2; } b2rt_point_query;      /* 16 B */
typedef struct { float d2, u, v; uint32_t tri; } b2rt_point_hit;   /* 16 B */
int b2rt_closest_point(b2rt_context* ctx, const b2rt_point_query* q, uint64_t n, b2rt_point_hit* out);
int b2rt_closest_point_device(b2rt_context* ctx, const b2rt_point_query* d_q, uint64_t n, b2rt_point_hit* d_out, void* cuda_stream);

/* ---- path-traced radiance (new) ------------------------------------------------------------ */
/* Render() (kernel_bvh.cl:349-384) started from a caller's ray instead of the pinhole camera: one shaded sample per ray, for
 * other cameras (fisheye, orthographic, thin lens, panoramas), own sample patterns, probes at arbitrary points.
 *  Path i starts at InitRay((ox,oy,oz), (dx,dy,dz)) of rays[i] with RNG state seeds[i].
 *  Segment 0 is the closest hit with isect.t = tmax, under the acceptance rule of b2rt_trace_closest (tmin ignored, front
 *    faces only); a miss within tmax takes the sky term. Later segments start at pos + wi*0.01 with B2RT_MAX_RENDER_DIST,
 *    exactly as Render() does: with tmax = 100000 the whole path is Render().
 *  Shading arguments come from the bound slots LIGHT_BOUNCES (8), LIGHT_TYPE (9) and SKYBOX_INTENSITY (10) and the material
 *    buffer (slot 3); an out-of-range mtlIndex takes the last material, as in frames. The frame-only slots (output image,
 *    width, height, frame count, camera) are not needed.
 *  out[i] = {max(radiance, 0) per channel (OpenCL max: NaN passes), RNG state after the path}. The returned state lets a
 *    caller chain samples of one path. bounces <= 0 gives {0, 0, 0, seeds[i]}.
 *  A NULL rays, seeds or out with n > 0 returns B2RT_INVALID_VALUE and writes nothing; n = 0 succeeds. Slots 8-10 never
 *    set, no bound material buffer or no scene return B2RT_INVALID_KERNEL_ARGS.
 * b2rt_trace_radiance: host buffers, synchronous, pipelined in chunks like b2rt_trace_closest; on a b2rt_create_multi handle
 * the rays are cut into contiguous ranges, one per device.
 * b2rt_trace_radiance_device: device buffers, asynchronous on cuda_stream (NULL = the context's stream); on a
 * b2rt_create_multi handle it runs on the root. The launch uses the frame path's wavefront queues, so it runs on the
 * context's stream, ordered after the work already enqueued on cuda_stream, and work enqueued on cuda_stream after the call
 * sees the records (also after a failure, which may leave part of d_out written). Frames and radiance launches on
 * different streams are therefore serialised through the context's stream and never share the queues concurrently.
 * B2RT_OPT_TRAVERSAL = 1 runs one thread per path over the reference-layout arrays, B2RT_OPT_COUNTERS = 1 the counting build
 * (rays = path segments traced). B2RT_OPT_WAVEFRONT_LANES, B2RT_OPT_COOP_MAX and B2RT_OPT_RESUME_MAX apply as in frames;
 * B2RT_OPT_RENDER_MODE is ignored. Results do not depend on any of them. */
typedef struct { float r, g, b; uint32_t seed; } b2rt_radiance;          /* 16 B */
int b2rt_trace_radiance(b2rt_context* ctx, const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out);
int b2rt_trace_radiance_device(b2rt_context* ctx, const b2rt_ray* d_rays, const uint32_t* d_seeds, uint64_t n,
                               b2rt_radiance* d_out, void* cuda_stream);

/* CreateRay (kernel_bvh.cl:386-403) for gid in [gid_begin, gid_end) with the currently bound
 * WIDTH/HEIGHT/FRAME_COUNT/CAMERA_* arguments, written to device memory as b2rt_ray. */
int b2rt_camera_rays_device(b2rt_context* ctx, size_t gid_begin, size_t gid_end, b2rt_ray* d_rays, void* cuda_stream);

/* ---- multi-GPU (new; SURVEY.md 8e) ----------------------------------------------------------- */
/* ONE handle that drives n devices of this process. The reference creates its context over all devices of platform 0
 * (CLutils.cpp:20-26) but binds the queue to device 0 (CLutils.cpp:29); here every entry point really fans out:
 *  - buffers created with host data are uploaded to device_ids[0] (the root) and broadcast to the others over NVLink
 *    (ncclBroadcast); the compressed wide BVH is built once and broadcast likewise;
 *  - b2rt_execute / b2rt_execute_range deal 8-row bands of gid = y*W + x (kernel_bvh.cl:394-395) round robin to the
 *    devices; each device keeps the running average of ITS pixels and stores every finished pixel through to the root's
 *    image over a peer mapping, so b2rt_read_buffer / b2rt_read_pixels after it return the complete frame (the root's
 *    stream waits for all devices);
 *  - b2rt_trace_closest / b2rt_trace_any / b2rt_trace_multi cut the host ray stream into contiguous ranges, one per device,
 *    and b2rt_closest_point its queries likewise;
 *  - the *_device entry points, b2rt_build_bvh and b2rt_execute_bands address one device: the root
 *    (b2rt_build_scene_device builds there and copies the scene to every device).
 * n_devices == 1 gives an ordinary handle. CLRaytracer code written against the single-device calls runs unchanged. */
int b2rt_create_multi(const int* device_ids, int n_devices, b2rt_context** out);
/* Devices behind a handle (b2rt_create_multi), or ranks of its job (b2rt_comm_init); 1 otherwise. */
int b2rt_group_size(const b2rt_context* ctx);
/* peer_store: finished pixels reach the root's image by direct stores over NVLink (else by copies / send-recv);
 * nccl_loaded: NCCL was found at run time (dlopen "libnccl.so.2"). Either pointer may be NULL. */
int b2rt_group_info(const b2rt_context* ctx, int* peer_store, int* nccl_loaded);

/* One process per GPU (e.g. torchrun): the same partition, every rank with its own single-device handle and scene.
 * b2rt_comm_unique_id: on one rank; distribute the bytes (>= 128) to all ranks by any means. b2rt_comm_init: collective,
 * creates the NCCL communicator. b2rt_comm_share_output: collective, after every rank has bound an output image of the
 * same size (b2rt_resize): rank 0's image is mapped into the other ranks (CUDA IPC handle broadcast over NCCL) as their
 * store-through target. b2rt_execute_shard: KernelEntry for this rank's bands of the WIDTH x HEIGHT frame, then the
 * gather on rank 0 -- a 4-byte ncclAllReduce as completion barrier when the image is mapped (pixels were stored through
 * by the kernels), else grouped ncclSend/ncclRecv of the bands straight into place. Asynchronous: rank 0 reads the
 * complete frame with b2rt_read_pixels + b2rt_finish. Rank 0's stream is the reference point of the image: the next
 * b2rt_execute_shard on any rank starts storing only after rank 0's stream has reached ITS next b2rt_execute_shard, i.e.
 * after the reads rank 0 enqueued in between (entry fence, B2RT_OPT_SHARD_FENCE). A device-group handle
 * (b2rt_create_multi) orders its peers behind the root's stream the same way, with an event. */
int b2rt_comm_unique_id(void* id_out, size_t bytes);
int b2rt_comm_init(b2rt_context* ctx, const void* id, size_t bytes, int rank, int world);
int b2rt_comm_share_output(b2rt_context* ctx);
int b2rt_execute_shard(b2rt_context* ctx);
/* The partition itself (no device needed): rank's n_full_bands whole bands of band_pixels gids start at gid_begin and
 * are stride_pixels apart; [tail_begin, tail_end) is the frame's clipped last band if this rank owns it (else empty). */
int b2rt_shard_bands(uint32_t width, uint32_t height, int rank, int world, uint64_t* gid_begin, uint32_t* band_pixels,
                     uint32_t* stride_pixels, uint32_t* n_full_bands, uint64_t* tail_begin, uint64_t* tail_end);

/* ---- introspection -------------------------------------------------------------------- */
int b2rt_device_pointer(b2rt_context* ctx, b2rt_buffer buf, void** d_ptr, size_t* bytes);
int b2rt_bound_buffer(b2rt_context* ctx, uint32_t slot, b2rt_buffer* out);
int b2rt_scene_info_get(b2rt_context* ctx, b2rt_scene_info* out);
int b2rt_set_option(b2rt_context* ctx, uint32_t option, int64_t value);
int b2rt_get_counters(b2rt_context* ctx, b2rt_counters* out);   /* accumulated since reset */
int b2rt_reset_counters(b2rt_context* ctx);
/* Stage durations of the LAST wavefront frame launch made with B2RT_OPT_STAGE_TIMES = 1 (waits for it): kinds[i] is a
 * B2RT_STAGE_* code, ms[i] the time between the end of the previous stage and the end of this one on the device. */
enum { B2RT_STAGE_BEGIN = 0, B2RT_STAGE_GENERATE = 1, B2RT_STAGE_TRACE = 2, B2RT_STAGE_TAIL = 3, B2RT_STAGE_SHADE = 4 };
int b2rt_stage_times(b2rt_context* ctx, uint32_t* kinds, float* ms, uint32_t capacity, uint32_t* n_out);
/* Kernels launched by this context since creation (for bench.py's gpu_launches). */
uint64_t b2rt_launch_count(const b2rt_context* ctx);
int b2rt_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B2RT_H */
