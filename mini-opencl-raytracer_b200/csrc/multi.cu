// multi.cu -- multi-GPU behind the C ABI (SURVEY.md 8e): the scene is replicated, screen bands (gid = y*W + x,
// kernel_bvh.cl:394-395) and ray ranges are dealt to the GPUs, and the frame is gathered on the root GPU.
//
//  * b2rt_create_multi: ONE handle that drives n devices of this process -- what the reference's context over "all
//    devices of platform 0" (CLutils.cpp:20-26) never did (its queue is bound to device 0). Every entry point fans out:
//    buffers with host data are uploaded once and broadcast root -> peers over NVLink (ncclBroadcast; cudaMemcpyPeer when
//    NCCL cannot be loaded), the compressed wide BVH is built once and broadcast, b2rt_execute splits the frame into
//    8-row bands dealt round robin, ray streams are cut into contiguous ranges. One host thread per peer issues its
//    launches, so launch latency does not add up over the devices.
//  * b2rt_comm_*: the same partition for one-process-per-GPU jobs (torchrun): an NCCL communicator created from a
//    caller-distributed unique id; b2rt_execute_shard renders this rank's bands.
//  * Gather: the ranks' shade / megakernel epilogue stores every finished pixel straight into the root's image through a
//    peer mapping (cudaDeviceEnablePeerAccess, or a CUDA IPC handle exchanged over NCCL between processes), see
//    accumulate() in shade.cuh -- compute and gather are one kernel; what remains of the collective is a completion
//    barrier (events inside a process, a 4-byte ncclAllReduce between processes). Without peer access the bands travel
//    by grouped ncclSend/ncclRecv (or a strided peer copy inside a process) straight into place: bands are contiguous in
//    the image, so nothing is packed or unpacked.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): inside a PyTorch process that is the library torch already loaded,
// in a plain C++ program the system's.
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <thread>
#include "context.h"

using namespace b2rt;
using namespace b2rt_detail;

namespace b2rt_detail {

// ---- NCCL, bound at run time --------------------------------------------------------------------------------------
struct Nccl {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    std::string error;
};

static Nccl* nccl() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, []() {
        for (const char* name : { "libnccl.so.2", "libnccl.so" }) {
            n.lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (n.lib) break;
        }
        if (!n.lib) { n.error = std::string("NCCL not loadable: ") + dlerror(); return; }
        bool ok = true;
        auto bind = [&](auto& fn, const char* sym) { fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(n.lib, sym)); if (!fn) { ok = false; n.error = std::string("NCCL symbol missing: ") + sym; } };
        bind(n.GetUniqueId, "ncclGetUniqueId"); bind(n.CommInitRank, "ncclCommInitRank"); bind(n.CommInitAll, "ncclCommInitAll");
        bind(n.CommDestroy, "ncclCommDestroy"); bind(n.Broadcast, "ncclBroadcast"); bind(n.AllReduce, "ncclAllReduce");
        bind(n.Send, "ncclSend"); bind(n.Recv, "ncclRecv"); bind(n.GroupStart, "ncclGroupStart"); bind(n.GroupEnd, "ncclGroupEnd");
        bind(n.GetErrorString, "ncclGetErrorString");
        if (!ok) { dlclose(n.lib); n.lib = nullptr; }
    });
    return n.lib ? &n : nullptr;
}

static int nccl_fail(b2rt_context* ctx, ncclResult_t r, const char* what) {
    Nccl* n = nccl();
    return fail(ctx, B2RT_OUT_OF_RESOURCES, std::string(what) + ": " + (n ? n->GetErrorString(r) : "NCCL unavailable"));
}
#define NK(call)                                                          \
    do {                                                                  \
        ncclResult_t r__ = (call);                                        \
        if (r__ != ncclSuccess) return nccl_fail(ctx, r__, #call);        \
    } while (0)

// ---- band partition -------------------------------------------------------------------------------------------------
// Work items [begin, end) cut into bands of `band` items dealt round robin to `world` ranks: rank k owns bands k, k+world,
// ...; n_full of them are whole, and at most one rank owns the clipped last band [tail_begin, tail_end).
struct BandShare { uint64_t first = 0; uint32_t band = 0, stride = 0, n_full = 0; uint64_t tail_begin = 0, tail_end = 0; };

static BandShare band_share(uint64_t begin, uint64_t end, uint64_t band, int rank, int world) {
    BandShare s;
    s.band = (uint32_t)band;
    s.stride = (uint32_t)(band * (uint64_t)world);
    s.first = begin + (uint64_t)rank * band;
    const uint64_t n = end - begin, whole = n / band, rest = n % band;
    s.n_full = whole > (uint64_t)rank ? (uint32_t)((whole - rank + world - 1) / world) : 0u;
    if (rest && whole % (uint64_t)world == (uint64_t)rank) { s.tail_begin = begin + whole * band; s.tail_end = end; }
    return s;
}

static int render_share(b2rt_context* ctx, const BandShare& s) {
    if (s.n_full) {
        GidMap map;
        map.begin = s.first; map.band = s.band; map.stride = s.stride;
        int st = render_items(ctx, map, (uint64_t)s.band * s.n_full);
        if (st) return st;
    }
    if (s.tail_end > s.tail_begin) {
        GidMap map;
        map.begin = s.tail_begin; map.band = map.stride = (uint32_t)(s.tail_end - s.tail_begin);
        return render_items(ctx, map, s.tail_end - s.tail_begin);
    }
    return B2RT_SUCCESS;
}

static uint64_t band_items(const b2rt_context* ctx) {
    const uint64_t rows = 8;                                   // 8-row bands: sky and geometry rows interleave over the ranks
    return ctx->width ? rows * ctx->width : 4096;
}

// ---- one handle, several devices of this process -------------------------------------------------------------------
struct Worker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, done = false, quit = false;
    int result = 0;
    void loop() {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            std::function<int()> j = std::move(job);
            has_job = false;
            lk.unlock();
            int r = j();
            lk.lock();
            result = r; done = true;
            cv.notify_all();
        }
    }
    void post(std::function<int()> j) { std::lock_guard<std::mutex> lk(m); job = std::move(j); has_job = true; done = false; cv.notify_all(); }
    int wait() { std::unique_lock<std::mutex> lk(m); cv.wait(lk, [&] { return done; }); return result; }
};

struct Group {
    std::vector<b2rt_context*> members;                  // [0] is the handle itself (the root: it holds the complete frame)
    std::vector<std::unique_ptr<Worker>> workers;       // [k-1] issues member k's work
    std::vector<ncclComm_t> comms;                       // empty when NCCL could not be loaded
    std::vector<cudaEvent_t> done;                       // member k's share of the frame has been rendered
    cudaEvent_t root_free = nullptr;                     // the root's stream has reached this frame: earlier reads of its image are done
    bool peer_store = false;                             // every member can store into the root's memory
};

// fn(member) on every member, the peers on their own threads. First failure wins; its text is copied to the handle.
static int run_members(b2rt_context* root, const std::function<int(b2rt_context*, int)>& fn) {
    Group* g = root->group;
    const int n = (int)g->members.size();
    for (int k = 1; k < n; ++k) { b2rt_context* m = g->members[k]; g->workers[k - 1]->post([&fn, m, k]() { return fn(m, k); }); }
    int st = fn(root, 0);
    for (int k = 1; k < n; ++k) {
        int r = g->workers[k - 1]->wait();
        if (r && !st) { st = r; root->error = "device " + std::to_string(g->members[k]->device) + ": " + g->members[k]->error; }
    }
    return st;
}

// The same `bytes` from the root's pointer to every peer's (ptrs[k] on member k), ordered on the members' streams.
static int broadcast(b2rt_context* ctx, void* const* ptrs, size_t bytes) {
    Group* g = ctx->group;
    const int n = (int)g->members.size();
    if (bytes == 0 || n < 2) return B2RT_SUCCESS;
    Nccl* nc = nccl();
    if (nc && !g->comms.empty()) {
        NK(nc->GroupStart());
        for (int k = 0; k < n; ++k) {
            ncclResult_t r = nc->Broadcast(ptrs[0], ptrs[k], bytes, ncclChar, 0, g->comms[k], g->members[k]->stream);
            if (r != ncclSuccess) { nc->GroupEnd(); return nccl_fail(ctx, r, "ncclBroadcast"); }
        }
        NK(nc->GroupEnd());
    } else {
        CK(cudaSetDevice(ctx->device));
        for (int k = 1; k < n; ++k)
            CK(cudaMemcpyPeerAsync(ptrs[k], g->members[k]->device, ptrs[0], ctx->device, bytes, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    for (int k = 0; k < n; ++k) {
        CK(cudaSetDevice(g->members[k]->device));
        CK(cudaStreamSynchronize(g->members[k]->stream));
    }
    CK(cudaSetDevice(ctx->device));
    return B2RT_SUCCESS;
}

int group_buffer_create(b2rt_context* ctx, uint32_t flags, size_t bytes, const void* host_ptr, b2rt_buffer* out) {
    Group* g = ctx->group;
    int st = buffer_create_single(ctx, flags, bytes, host_ptr, out, true);
    if (st) return st;
    std::vector<void*> ptrs{ find(ctx, *out)->d_ptr };
    for (size_t k = 1; k < g->members.size(); ++k) {
        b2rt_context* m = g->members[k];
        b2rt_buffer id = 0;
        // peers receive host data from the root over NVLink; buffers without host data are zero-filled like the root's
        st = buffer_create_single(m, flags & ~(uint32_t)B2RT_MEM_COPY_HOST_PTR, bytes, nullptr, &id, host_ptr == nullptr);
        if (st) return fail(ctx, st, "device " + std::to_string(m->device) + ": " + m->error);
        if (id != *out) return fail(ctx, B2RT_OUT_OF_RESOURCES, "buffer ids of the device group went out of step");
        ptrs.push_back(find(m, id)->d_ptr);
    }
    if (host_ptr) return broadcast(ctx, ptrs.data(), bytes);
    return B2RT_SUCCESS;
}

int group_broadcast_buffer(b2rt_context* ctx, b2rt_buffer id) {
    Group* g = ctx->group;
    Buffer* b = find(ctx, id);
    if (!b) return fail(ctx, B2RT_INVALID_MEM_OBJECT, "unknown buffer");
    std::vector<void*> ptrs{ b->d_ptr };
    for (size_t k = 1; k < g->members.size(); ++k) {
        Buffer* p = find(g->members[k], id);
        if (!p || p->bytes != b->bytes) return fail(ctx, B2RT_OUT_OF_RESOURCES, "buffer ids of the device group went out of step");
        ptrs.push_back(p->d_ptr);
    }
    return broadcast(ctx, ptrs.data(), b->bytes);
}

int group_each(b2rt_context* ctx, int (*fn)(b2rt_context*, void*), void* arg, bool parallel) {
    Group* g = ctx->group;
    if (parallel) return run_members(ctx, [fn, arg](b2rt_context* m, int) { return fn(m, arg); });
    for (b2rt_context* m : g->members) {
        int st = fn(m, arg);
        if (st) { if (m != ctx) ctx->error = "device " + std::to_string(m->device) + ": " + m->error; return st; }
    }
    return B2RT_SUCCESS;
}

// Peers store finished pixels into the root's image (slot 0) when it is peer-mapped.
void group_bind_output(b2rt_context* ctx) {
    Group* g = ctx->group;
    Buffer* out = find(ctx, ctx->bound[B2RT_ARG_BUFFER_OUT]);
    for (size_t k = 1; k < g->members.size(); ++k)
        g->members[k]->mirror = (g->peer_store && out) ? static_cast<float*>(out->d_ptr) : nullptr;
}

// The root has just built and uploaded the compressed wide BVH: the peers take copies over NVLink.
int group_adopt_scene(b2rt_context* root) {
    Group* g = root->group;
    const size_t wb = std::max<size_t>(root->info.wide_node_bytes, sizeof(WideNode)), lb = std::max<size_t>(root->info.leaf_bytes, 16) + 64,
                 sb = std::max<size_t>(root->info.shading_bytes, 48);
    const size_t cb = std::max<size_t>(root->info.n_wide_nodes * 32, 32), db = std::max<size_t>(root->info.n_leaf_blocks * 8, 8);
    std::vector<void*> pw{ root->d_wide }, pl{ root->d_leaf }, ps{ root->d_shade }, pc{ root->d_child_bin }, pd{ root->d_leaf_dir };
    for (size_t k = 1; k < g->members.size(); ++k) {
        b2rt_context* ctx = g->members[k];
        CK(cudaSetDevice(ctx->device));
        free_scene(ctx);
        free_tail(ctx);
        int st_alloc = alloc_bvh(ctx, root->info.wide_node_bytes, root->info.leaf_bytes);
        if (st_alloc) return st_alloc;
        CK(cudaMalloc(&ctx->d_shade, sb));
        CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_child_bin), cb));
        CK(cudaMalloc(reinterpret_cast<void**>(&ctx->d_leaf_dir), db));
        pw.push_back(ctx->d_wide); pl.push_back(ctx->d_leaf); ps.push_back(ctx->d_shade); pc.push_back(ctx->d_child_bin); pd.push_back(ctx->d_leaf_dir);
    }
    b2rt_context* ctx = root;
    CK(cudaSetDevice(root->device));
    int st = broadcast(root, pw.data(), wb);
    if (!st) st = broadcast(root, pl.data(), lb);
    if (!st) st = broadcast(root, ps.data(), sb);
    if (!st) st = broadcast(root, pc.data(), cb);
    if (!st) st = broadcast(root, pd.data(), db);
    if (st) return st;
    for (size_t k = 1; k < g->members.size(); ++k) {
        b2rt_context* m = g->members[k];
        Buffer *bt = find(m, m->bound[B2RT_ARG_BUFFER_SCENE]), *bn = find(m, m->bound[B2RT_ARG_BUFFER_NODE]), *bm = find(m, m->bound[B2RT_ARG_BUFFER_MATERIAL]);
        if (!bt || !bn) return fail(root, B2RT_INVALID_KERNEL_ARGS, "device group: scene buffers are not bound on every device");
        m->info = root->info;
        m->stack_bound = root->stack_bound;
        m->view = root->view;
        m->view.wide = static_cast<const U4*>(m->d_wide);
        m->view.leaf = static_cast<const U4*>(m->d_leaf);
        m->view.shade = static_cast<const ShadeTri*>(m->d_shade);
        m->view.mats = bm ? static_cast<const RefMaterial*>(bm->d_ptr) : nullptr;
        m->view.tris = static_cast<const RefTriangle*>(bt->d_ptr);
        m->view.nodes = static_cast<const RefNode*>(bn->d_ptr);
        m->grid_closest = root->grid_closest / std::max(root->sm_count, 1) * m->sm_count;
        m->grid_any = root->grid_any / std::max(root->sm_count, 1) * m->sm_count;
        m->grid_tail = root->grid_tail / std::max(root->sm_count, 1) * m->sm_count;
        m->tail_rec_words = root->tail_rec_words;
        m->tail_capacity_records = root->tail_capacity_records / std::max(root->sm_count, 1) * m->sm_count;
        m->tuner.clear();
        m->tune_pending_mode = -1;
        m->scene_dirty = false;
        cudaSetDevice(m->device);
        scene_l2_setup(m);
    }
    cudaSetDevice(root->device);
    return B2RT_SUCCESS;
}

// KernelEntry for gid in [gid_begin, gid_end) on all devices: 8-row bands dealt round robin, each member one strided
// launch sequence; the root's stream then waits for every member, so a read of the image enqueued next sees all of it.
int group_execute(b2rt_context* ctx, size_t gid_begin, size_t gid_end) {
    Group* g = ctx->group;
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);                              // builds once, peers adopt
    if (st) return st;
    const int world = (int)g->members.size();
    const uint64_t band = band_items(ctx);
    // The peers write into the root's image (store-through or band copies). Whatever the root's stream still has to do with
    // that image -- an asynchronous b2rt_read_buffer of the previous frame above all -- must come first: without this
    // edge a peer's pixels of frame f+1 could land in the middle of the read of frame f.
    CK(cudaEventRecord(g->root_free, ctx->stream));
    st = run_members(ctx, [&](b2rt_context* m, int k) {
        int s = use_device(m);
        if (s) return s;
        if (k) { b2rt_context* ctx = m; CK(cudaStreamWaitEvent(m->stream, g->root_free, 0)); }
        s = render_share(m, band_share(gid_begin, gid_end, band, k, world));
        if (s || k == 0) return s;
        b2rt_context* ctx = m;
        const BandShare sh = band_share(gid_begin, gid_end, band, k, world);
        if (!g->peer_store) {
            // no peer mapping: copy this member's bands into place in the root's image (one strided copy + the clipped band)
            Buffer *src = find(m, m->bound[0]), *dst = find(g->members[0], g->members[0]->bound[0]);
            if (src && dst && sh.n_full)
                CK(cudaMemcpy2DAsync(static_cast<char*>(dst->d_ptr) + sh.first * 16, (size_t)sh.stride * 16, static_cast<char*>(src->d_ptr) + sh.first * 16,
                                     (size_t)sh.stride * 16, (size_t)sh.band * 16, sh.n_full, cudaMemcpyDefault, m->stream));
            if (src && dst && sh.tail_end > sh.tail_begin)
                CK(cudaMemcpyAsync(static_cast<char*>(dst->d_ptr) + sh.tail_begin * 16, static_cast<char*>(src->d_ptr) + sh.tail_begin * 16,
                                   (sh.tail_end - sh.tail_begin) * 16, cudaMemcpyDefault, m->stream));
        }
        CK(cudaEventRecord(g->done[k], m->stream));
        return (int)B2RT_SUCCESS;
    });
    if (st) return st;
    CK(cudaSetDevice(ctx->device));
    for (int k = 1; k < world; ++k) CK(cudaStreamWaitEvent(ctx->stream, g->done[k], 0));
    return B2RT_SUCCESS;
}

int group_split(b2rt_context* ctx, uint64_t n, const std::function<int(b2rt_context*, uint64_t, uint64_t)>& fn) {
    Group* g = ctx->group;
    int st = use_device(ctx);
    if (st) return st;
    st = ensure_scene(ctx);
    if (st) return st;
    const uint64_t world = g->members.size();
    return run_members(ctx, [&](b2rt_context* m, int k) {
        const uint64_t lo = n * (uint64_t)k / world, hi = n * (uint64_t)(k + 1) / world;     // contiguous ranges, no collective
        if (hi == lo) return (int)B2RT_SUCCESS;
        return fn(m, lo, hi - lo);
    });
}

const std::vector<b2rt_context*>& group_members(const b2rt_context* ctx) { return ctx->group->members; }

int group_finish(b2rt_context* ctx) {
    return run_members(ctx, [](b2rt_context* ctx, int) {
        int st = use_device(ctx);
        if (st) return st;
        CK(cudaStreamSynchronize(ctx->stream));
        return (int)B2RT_SUCCESS;
    });
}

void group_destroy(b2rt_context* ctx) {
    Group* g = ctx->group;
    if (!g) return;
    for (auto& w : g->workers) {
        { std::lock_guard<std::mutex> lk(w->m); w->quit = true; w->cv.notify_all(); }
        if (w->th.joinable()) w->th.join();
    }
    Nccl* nc = nccl();
    for (size_t k = 0; k < g->comms.size(); ++k) if (nc && g->comms[k]) nc->CommDestroy(g->comms[k]);
    for (size_t k = 0; k < g->done.size(); ++k) if (g->done[k]) { cudaSetDevice(g->members[k]->device); cudaEventDestroy(g->done[k]); }
    if (g->root_free) { cudaSetDevice(ctx->device); cudaEventDestroy(g->root_free); }
    for (size_t k = 1; k < g->members.size(); ++k) { g->members[k]->parent = nullptr; b2rt_destroy(g->members[k]); }
    ctx->group = nullptr;
    delete g;
}

// ---- one process per GPU ----------------------------------------------------------------------------------------------
struct Comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    int* d_flag = nullptr;                               // completion barrier operand
    char* d_handle = nullptr;                            // 64-byte CUDA IPC handle in flight
    bool shared = false;                                 // the ranks store into rank 0's image through an IPC mapping
};

void comm_destroy(b2rt_context* ctx) {
    Comm* c = ctx->comm;
    if (!c) return;
    cudaSetDevice(ctx->device);
    if (ctx->mirror_ipc_base) { cudaIpcCloseMemHandle(ctx->mirror_ipc_base); ctx->mirror_ipc_base = nullptr; ctx->mirror = nullptr; }
    Nccl* nc = nccl();
    if (nc && c->comm) nc->CommDestroy(c->comm);
    if (c->d_flag) cudaFree(c->d_flag);
    if (c->d_handle) cudaFree(c->d_handle);
    ctx->comm = nullptr;
    delete c;
}

}  // namespace b2rt_detail

// ---- C ABI ---------------------------------------------------------------------------------------------------------------
extern "C" int b2rt_create_multi(const int* device_ids, int n_devices, b2rt_context** out) {
    if (!out) return fail(nullptr, B2RT_INVALID_VALUE, "null output handle");
    *out = nullptr;
    if (!device_ids || n_devices < 1 || n_devices > 64) return fail(nullptr, B2RT_INVALID_VALUE, "device list must name 1..64 devices");
    // B2RT_ALLOW_DUPLICATE_DEVICES=1 (tests on a one-GPU machine): the same device may be named several times; each mention
    // is a member with its own streams and buffers, which exercises the partition, the worker threads and the store-through
    const bool dup_ok = getenv("B2RT_ALLOW_DUPLICATE_DEVICES") != nullptr;
    for (int i = 0; i < n_devices && !dup_ok; ++i)
        for (int j = 0; j < i; ++j)
            if (device_ids[i] == device_ids[j]) return fail(nullptr, B2RT_INVALID_VALUE, "device " + std::to_string(device_ids[i]) + " named twice");
    b2rt_context* root = nullptr;
    int st = b2rt_create(device_ids[0], &root);
    if (st) return st;
    if (n_devices == 1) { *out = root; return B2RT_SUCCESS; }
    Group* g = new (std::nothrow) Group();
    if (!g) { b2rt_destroy(root); return fail(nullptr, B2RT_OUT_OF_HOST_MEMORY, "device group"); }
    root->group = g;
    g->members.push_back(root);
    auto bail = [&](int status, const std::string& msg) { b2rt_destroy(root); return fail(nullptr, status, msg); };
    for (int k = 1; k < n_devices; ++k) {
        b2rt_context* m = nullptr;
        st = b2rt_create(device_ids[k], &m);
        if (st) { std::string why = b2rt_last_error(nullptr); return bail(st, why); }
        m->parent = root;
        g->members.push_back(m);
    }
    // peer mappings: every member must be able to store into the root's memory for the fused gather
    g->peer_store = true;
    for (int k = 1; k < n_devices; ++k) {
        if (device_ids[k] == device_ids[0]) continue;            // same device: its memory is directly addressable
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, device_ids[k], device_ids[0]) != cudaSuccess || !can) { cudaGetLastError(); g->peer_store = false; continue; }
        cudaSetDevice(device_ids[k]);
        cudaError_t e = cudaDeviceEnablePeerAccess(device_ids[0], 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) g->peer_store = false;
        cudaGetLastError();
        // and the root reads the peers' memory in the copy fallback / broadcasts
        cudaSetDevice(device_ids[0]);
        e = cudaDeviceEnablePeerAccess(device_ids[k], 0);
        cudaGetLastError();
    }
    g->done.assign(n_devices, nullptr);
    for (int k = 0; k < n_devices; ++k) {
        cudaSetDevice(device_ids[k]);
        if (cudaEventCreateWithFlags(&g->done[k], cudaEventDisableTiming) != cudaSuccess) return bail(B2RT_OUT_OF_RESOURCES, "cudaEventCreate (device group)");
    }
    cudaSetDevice(device_ids[0]);
    if (cudaEventCreateWithFlags(&g->root_free, cudaEventDisableTiming) != cudaSuccess) return bail(B2RT_OUT_OF_RESOURCES, "cudaEventCreate (device group)");
    if (Nccl* nc = nccl()) {
        g->comms.assign(n_devices, nullptr);
        ncclResult_t r = nc->CommInitAll(g->comms.data(), n_devices, device_ids);
        if (r != ncclSuccess) { g->comms.clear(); }                 // broadcasts fall back to cudaMemcpyPeer
    }
    for (int k = 1; k < n_devices; ++k) {
        g->workers.emplace_back(new Worker());
        Worker* w = g->workers.back().get();
        w->th = std::thread([w]() { w->loop(); });
    }
    cudaSetDevice(device_ids[0]);
    *out = root;
    return B2RT_SUCCESS;
}

extern "C" int b2rt_group_size(const b2rt_context* ctx) {
    if (!ctx) return 0;
    if (ctx->group) return (int)ctx->group->members.size();
    return ctx->comm ? ctx->comm->world : 1;
}

extern "C" int b2rt_group_info(const b2rt_context* ctx, int* peer_store, int* nccl_loaded) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (peer_store) *peer_store = ctx->group ? (ctx->group->peer_store ? 1 : 0) : (ctx->comm ? (ctx->comm->shared ? 1 : 0) : 0);
    if (nccl_loaded) *nccl_loaded = ctx->group ? (ctx->group->comms.empty() ? 0 : 1) : (ctx->comm ? 1 : 0);
    return B2RT_SUCCESS;
}

extern "C" int b2rt_shard_bands(uint32_t width, uint32_t height, int rank, int world, uint64_t* gid_begin, uint32_t* band_pixels,
                                uint32_t* stride_pixels, uint32_t* n_full_bands, uint64_t* tail_begin, uint64_t* tail_end) {
    if (!width || !height || world < 1 || rank < 0 || rank >= world) return B2RT_INVALID_VALUE;
    const BandShare s = band_share(0, (uint64_t)width * height, 8ull * width, rank, world);
    if (gid_begin) *gid_begin = s.first;
    if (band_pixels) *band_pixels = s.band;
    if (stride_pixels) *stride_pixels = s.stride;
    if (n_full_bands) *n_full_bands = s.n_full;
    if (tail_begin) *tail_begin = s.tail_begin;
    if (tail_end) *tail_end = s.tail_end;
    return B2RT_SUCCESS;
}

extern "C" int b2rt_comm_unique_id(void* id_out, size_t bytes) {
    if (!id_out || bytes < sizeof(ncclUniqueId)) return fail(nullptr, B2RT_INVALID_VALUE, "unique id buffer must hold " + std::to_string(sizeof(ncclUniqueId)) + " bytes");
    Nccl* nc = nccl();
    if (!nc) return fail(nullptr, B2RT_OUT_OF_RESOURCES, "NCCL could not be loaded");
    ncclUniqueId id;
    ncclResult_t r = nc->GetUniqueId(&id);
    if (r != ncclSuccess) return nccl_fail(nullptr, r, "ncclGetUniqueId");
    memset(id_out, 0, bytes);
    memcpy(id_out, &id, sizeof(id));
    return B2RT_SUCCESS;
}

extern "C" int b2rt_comm_init(b2rt_context* ctx, const void* id, size_t bytes, int rank, int world) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    if (ctx->group || ctx->parent) return fail(ctx, B2RT_INVALID_VALUE, "a device-group handle cannot also be a rank of a multi-process job");
    if (ctx->comm) return fail(ctx, B2RT_INVALID_VALUE, "communicator already initialised");
    if (!id || bytes < sizeof(ncclUniqueId) || world < 1 || rank < 0 || rank >= world) return fail(ctx, B2RT_INVALID_VALUE, "bad communicator arguments");
    Nccl* nc = nccl();
    if (!nc) return fail(ctx, B2RT_OUT_OF_RESOURCES, "NCCL could not be loaded");
    int st = use_device(ctx);
    if (st) return st;
    Comm* c = new (std::nothrow) Comm();
    if (!c) return fail(ctx, B2RT_OUT_OF_HOST_MEMORY, "communicator");
    c->rank = rank; c->world = world;
    ctx->comm = c;
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    ncclResult_t r = nc->CommInitRank(&c->comm, world, uid, rank);
    if (r != ncclSuccess) { c->comm = nullptr; comm_destroy(ctx); return nccl_fail(ctx, r, "ncclCommInitRank"); }
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->d_flag), 256);
    if (e == cudaSuccess) e = cudaMemset(c->d_flag, 0, 256);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&c->d_handle), 256);
    if (e != cudaSuccess) { comm_destroy(ctx); return cuda_fail(ctx, e, "communicator scratch"); }
    return B2RT_SUCCESS;
}

// Collective: after every rank has bound its output image (b2rt_resize), rank 0's image becomes the store-through target
// of the others. Returns success with shared = false when the mapping is not possible (the gather then uses send/recv).
extern "C" int b2rt_comm_share_output(b2rt_context* ctx) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    Comm* c = ctx->comm;
    if (!c) return fail(ctx, B2RT_INVALID_VALUE, "b2rt_comm_init first");
    Nccl* nc = nccl();
    int st = use_device(ctx);
    if (st) return st;
    Buffer* out = find(ctx, ctx->bound[B2RT_ARG_BUFFER_OUT]);
    if (!out) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "output buffer (slot 0) is not bound");
    if (ctx->mirror_ipc_base) { cudaIpcCloseMemHandle(ctx->mirror_ipc_base); ctx->mirror_ipc_base = nullptr; }
    ctx->mirror = nullptr;
    c->shared = false;
    // message: [0] = 1 if a handle follows, [8..72) the handle, [72..80) the image size
    char msg[128];
    memset(msg, 0, sizeof(msg));
    if (c->rank == 0) {
        cudaIpcMemHandle_t h;
        if (cudaIpcGetMemHandle(&h, out->d_ptr) == cudaSuccess) { msg[0] = 1; memcpy(msg + 8, &h, sizeof(h)); }
        else cudaGetLastError();
        const uint64_t bytes = out->bytes;
        memcpy(msg + 72, &bytes, 8);
        CK(cudaMemcpyAsync(c->d_handle, msg, sizeof(msg), cudaMemcpyHostToDevice, ctx->stream));
    }
    NK(nc->Broadcast(c->d_handle, c->d_handle, sizeof(msg), ncclChar, 0, c->comm, ctx->stream));
    CK(cudaMemcpyAsync(msg, c->d_handle, sizeof(msg), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int ok = msg[0] == 1;
    uint64_t root_bytes = 0;
    memcpy(&root_bytes, msg + 72, 8);
    if (root_bytes != out->bytes) return fail(ctx, B2RT_INVALID_VALUE, "the ranks' output images differ in size");
    if (ok && c->rank != 0) {
        cudaIpcMemHandle_t h;
        memcpy(&h, msg + 8, sizeof(h));
        void* base = nullptr;
        if (cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess) { ctx->mirror_ipc_base = base; ctx->mirror = static_cast<float*>(base); }
        else { cudaGetLastError(); ok = 0; }
    }
    // everybody must agree: one rank without a mapping sends the whole job down the send/recv path
    int* flag = c->d_flag + 8;
    CK(cudaMemcpyAsync(flag, &ok, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    NK(nc->AllReduce(flag, flag, 1, ncclInt, ncclMin, c->comm, ctx->stream));
    CK(cudaMemcpyAsync(&ok, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (!ok) {
        if (ctx->mirror_ipc_base) { cudaIpcCloseMemHandle(ctx->mirror_ipc_base); ctx->mirror_ipc_base = nullptr; }
        ctx->mirror = nullptr;
    }
    c->shared = ok != 0;
    return B2RT_SUCCESS;
}

// This rank's share of KernelEntry over the WIDTH x HEIGHT frame, then the gather on rank 0 (asynchronous; rank 0's
// stream has the complete image after this call's work).
extern "C" int b2rt_execute_shard(b2rt_context* ctx) {
    if (!ctx) return B2RT_INVALID_CONTEXT;
    Comm* c = ctx->comm;
    if (!c) return fail(ctx, B2RT_INVALID_VALUE, "b2rt_comm_init first");
    Nccl* nc = nccl();
    int st = use_device(ctx);
    if (st) return st;
    if (!ctx->width || !ctx->height) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "WIDTH/HEIGHT must be non-zero");
    const uint64_t n = (uint64_t)ctx->width * ctx->height, band = band_items(ctx);
    if (c->world > 1 && c->shared && ctx->opt_shard_fence) {
        // Entry fence: nobody's kernels of THIS frame may store into rank 0's image before rank 0's stream has got here,
        // i.e. before whatever rank 0 enqueued after the previous frame's completion barrier -- its read of that frame --
        // is done. (The completion barrier alone does not give that: a rank leaves it as soon as everybody has joined.)
        NK(nc->AllReduce(c->d_flag + 16, c->d_flag + 16, 1, ncclInt, ncclSum, c->comm, ctx->stream));
    }
    st = render_share(ctx, band_share(0, n, band, c->rank, c->world));
    if (st) return st;
    if (c->world == 1) return B2RT_SUCCESS;
    if (c->shared) {
        // pixels are already in rank 0's image; what is left of the gather is "everybody's kernels have finished"
        NK(nc->AllReduce(c->d_flag, c->d_flag, 1, ncclInt, ncclSum, c->comm, ctx->stream));
        return B2RT_SUCCESS;
    }
    Buffer* out = find(ctx, ctx->bound[B2RT_ARG_BUFFER_OUT]);
    if (!out) return fail(ctx, B2RT_INVALID_KERNEL_ARGS, "output buffer (slot 0) is not bound");
    char* img = static_cast<char*>(out->d_ptr);
    NK(nc->GroupStart());
    ncclResult_t r = ncclSuccess;
    for (int k = 1; k < c->world && r == ncclSuccess; ++k) {
        if (c->rank != 0 && c->rank != k) continue;
        const BandShare s = band_share(0, n, band, k, c->world);
        for (uint32_t b = 0; b < s.n_full && r == ncclSuccess; ++b) {
            char* p = img + (s.first + (uint64_t)b * s.stride) * 16;
            r = c->rank == 0 ? nc->Recv(p, (size_t)s.band * 16, ncclChar, k, c->comm, ctx->stream) : nc->Send(p, (size_t)s.band * 16, ncclChar, 0, c->comm, ctx->stream);
        }
        if (s.tail_end > s.tail_begin && r == ncclSuccess) {
            char* p = img + s.tail_begin * 16;
            const size_t bytes = (s.tail_end - s.tail_begin) * 16;
            r = c->rank == 0 ? nc->Recv(p, bytes, ncclChar, k, c->comm, ctx->stream) : nc->Send(p, bytes, ncclChar, 0, c->comm, ctx->stream);
        }
    }
    ncclResult_t e = nc->GroupEnd();
    if (r != ncclSuccess) return nccl_fail(ctx, r, "ncclSend/ncclRecv (frame gather)");
    if (e != ncclSuccess) return nccl_fail(ctx, e, "ncclGroupEnd (frame gather)");
    return B2RT_SUCCESS;
}
