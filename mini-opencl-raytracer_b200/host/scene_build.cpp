// scene_build.cpp -- CLBounds3 helpers and CLBVHScene: the SAH BVH build + flattening that defines
// triangle order (= hit IDs) and the CLLinearBVHNode array the device consumes.
//
// Behavioural contract (reference CLBVHnode.cpp:7-207, CLmathlib.hpp:120-204): PBRT-style recursive
// build -- leaf when one primitive is left or all centroids coincide on the widest centroid axis;
// median split (std::nth_element) for two primitives; otherwise 12 centroid buckets, SAH cost
// 1 + (n0*A0 + n1*A1)/A, split (std::partition) when n > maxPrimitivesInNode or the best cost beats
// the leaf cost n. The arrays must come out IDENTICAL to the reference's (tests compare them with
// the verbatim reference build), because hit IDs are indices into the re-ordered triangle array. Two
// details of the reference matter for that and are reproduced on purpose:
//   * all arithmetic is fp32 in the reference's expression order (bucket index = int(12 * offset),
//     cost accumulation with int*float products, NaN costs from empty buckets never win `<`);
//   * the reference builds its two children inside one call expression,
//     InitInterior(dim, RecursiveBuild(first...), RecursiveBuild(second...)) (CLBVHnode.cpp:150-154);
//     g++ evaluates those arguments right to left, so the SECOND child's subtree is built -- and its
//     triangles appended to the ordered array -- before the first child's. Node numbering is still
//     pre-order with the first child at index+1 (CLBVHnode.cpp:161-183).
// Here the build writes an index-linked node pool with explicit work stacks (no per-node `new`, no recursion),
// builds independent subtrees of large scenes on a team of threads (B2RT_BUILD_THREADS, default all cores; the
// result does not depend on the thread count), then replays the reference's leaf emission order and numbers the
// nodes in pre-order.
#include <algorithm>
#include <atomic>
#include <cassert>
#include <cmath>
#include <cstdlib>
#include <limits>
#include <thread>
#include "glaze3d.h"

namespace Glaze3D
{
    // ---- CLBounds3 -----------------------------------------------------------------------------
    CLBounds3::CLBounds3()
    {
        const float hi = std::numeric_limits<float>::max(), lo = std::numeric_limits<float>::lowest();
        min = float3(hi, hi, hi);
        max = float3(lo, lo, lo);
    }
    static inline float3 lower(const float3& a, const float3& b) { return float3(std::min(a.x, b.x), std::min(a.y, b.y), std::min(a.z, b.z)); }
    static inline float3 upper(const float3& a, const float3& b) { return float3(std::max(a.x, b.x), std::max(a.y, b.y), std::max(a.z, b.z)); }
    CLBounds3::CLBounds3(const float3& a, const float3& b) : min(lower(a, b)), max(upper(a, b)) {}
    CLBounds3 Union(const CLBounds3& b, const float3& p) { CLBounds3 r; r.min = lower(b.min, p); r.max = upper(b.max, p); return r; }
    CLBounds3 Union(const CLBounds3& a, const CLBounds3& b) { CLBounds3 r; r.min = lower(a.min, b.min); r.max = upper(a.max, b.max); return r; }
    unsigned int CLBounds3::MaximumExtent() const
    {
        float3 d = Diagonal();
        if (d.x > d.y && d.x > d.z) return 0;
        return d.y > d.z ? 1 : 2;
    }
    float3 CLBounds3::Offset(const float3& p) const
    {
        float3 o = p - min;
        if (max.x > min.x) o.x /= max.x - min.x;
        if (max.y > min.y) o.y /= max.y - min.y;
        if (max.z > min.z) o.z /= max.z - min.z;
        return o;
    }

    void CLCamera::Update()
    {
        // CLcamera.h:15-21: `right` is refreshed from the OLD front before front is recomputed.
        right = vec3(front.y * up.z - front.z * up.y, front.z * up.x - front.x * up.z, front.x * up.y - front.y * up.x);
        front = vec3(std::cos(yaw) * std::sin(pitch), std::sin(yaw) * std::sin(pitch), std::cos(pitch));
    }

    // ---- BVH build ---------------------------------------------------------------------------------
    namespace
    {
        struct PrimInfo { unsigned int prim; CLBounds3 bounds; float3 centroid; };
        struct BuildNode { CLBounds3 bounds; int child[2]; int axis; unsigned int firstPrim, nPrims; };
        struct Bucket { int count = 0; CLBounds3 bounds; };
        constexpr unsigned int kBuckets = 12;

        struct Builder
        {
            std::vector<PrimInfo> info;
            std::vector<BuildNode> pool;
            std::vector<unsigned int> order;      // order[k] = original index of the k-th triangle of the new array
            unsigned int maxPrims = 0;

            int bucketOf(const CLBounds3& cb, unsigned int dim, const float3& centroid) const
            {
                int b = kBuckets * cb.Offset(centroid)[dim];     // unsigned * float -> float -> int, as in the reference
                if (b == (int)kBuckets) b = kBuckets - 1;
                assert(b >= 0 && b < (int)kBuckets);
                return b;
            }

            // A leaf remembers its range of `info`; the triangle order is emitted afterwards by emitOrder().
            static void makeLeaf(BuildNode& n, unsigned int start, unsigned int end, const CLBounds3& bounds)
            {
                n.firstPrim = start;
                n.nPrims = end - start;
                n.bounds = bounds;
                n.child[0] = n.child[1] = -1;
            }

            // Decides what `node` over info[start,end) is. Returns true and sets mid/dim for an interior node.
            // Touches only `node` and info[start,end), so disjoint ranges can be split concurrently.
            bool split(BuildNode& node, unsigned int start, unsigned int end, unsigned int& mid, unsigned int& dim)
            {
                CLBounds3 bounds;
                for (unsigned int i = start; i < end; ++i) bounds = Union(bounds, info[i].bounds);
                const unsigned int n = end - start;
                if (n == 1) { makeLeaf(node, start, end, bounds); return false; }
                CLBounds3 cb;
                for (unsigned int i = start; i < end; ++i) cb = Union(cb, info[i].centroid);
                dim = cb.MaximumExtent();
                mid = (start + end) / 2;
                if (cb.max[dim] == cb.min[dim]) { makeLeaf(node, start, end, bounds); return false; }
                if (n <= 2)
                {
                    const unsigned int d = dim;
                    std::nth_element(&info[start], &info[mid], &info[end - 1] + 1,
                                     [d](const PrimInfo& a, const PrimInfo& b) { return a.centroid[d] < b.centroid[d]; });
                }
                else
                {
                    Bucket buckets[kBuckets];
                    for (unsigned int i = start; i < end; ++i)
                    {
                        int b = bucketOf(cb, dim, info[i].centroid);
                        buckets[b].count++;
                        buckets[b].bounds = Union(buckets[b].bounds, info[i].bounds);
                    }
                    float cost[kBuckets - 1];
                    for (unsigned int i = 0; i < kBuckets - 1; ++i)
                    {
                        CLBounds3 b0, b1;
                        int c0 = 0, c1 = 0;
                        for (unsigned int j = 0; j <= i; ++j) { b0 = Union(b0, buckets[j].bounds); c0 += buckets[j].count; }
                        for (unsigned int j = i + 1; j < kBuckets; ++j) { b1 = Union(b1, buckets[j].bounds); c1 += buckets[j].count; }
                        cost[i] = 1.0f + (c0 * b0.SurfaceArea() + c1 * b1.SurfaceArea()) / bounds.SurfaceArea();
                    }
                    float best = cost[0];
                    unsigned int bestBucket = 0;
                    for (unsigned int i = 1; i < kBuckets - 1; ++i)
                        if (cost[i] < best) { best = cost[i]; bestBucket = i; }
                    if (!(n > maxPrims || best < float(n))) { makeLeaf(node, start, end, bounds); return false; }
                    const CLBounds3 cbv = cb;
                    const unsigned int d = dim;
                    PrimInfo* p = std::partition(&info[start], &info[end - 1] + 1, [=](const PrimInfo& pi) {
                        int b = kBuckets * cbv.Offset(pi.centroid)[d];
                        if (b == (int)kBuckets) b = kBuckets - 1;
                        return (unsigned int)b <= bestBucket;
                    });
                    mid = (unsigned int)(p - &info[0]);
                }
                return true;
            }

            struct Task { int id; unsigned int start, end; };

            // Splits `t` inside `nodes`; on an interior node appends the two children and returns their tasks.
            bool expand(std::vector<BuildNode>& nodes, const Task& t, Task& first, Task& second)
            {
                unsigned int mid = 0, dim = 0;
                BuildNode node = BuildNode();
                if (!split(node, t.start, t.end, mid, dim)) { nodes[t.id] = node; return false; }
                int c = (int)nodes.size();
                nodes.push_back(BuildNode());
                nodes.push_back(BuildNode());
                BuildNode& n = nodes[t.id];
                n.child[0] = c; n.child[1] = c + 1; n.axis = (int)dim; n.nPrims = 0; n.firstPrim = 0;
                first = Task{ c, t.start, mid };
                second = Task{ c + 1, mid, t.end };
                return true;
            }

            // Whole subtree of `root` (a task whose node already exists in `nodes`), depth-first.
            void buildSubtree(std::vector<BuildNode>& nodes, const Task& root)
            {
                std::vector<Task> todo;
                todo.push_back(root);
                while (!todo.empty())
                {
                    Task t = todo.back(), a, b;
                    todo.pop_back();
                    if (!expand(nodes, t, a, b)) continue;
                    todo.push_back(a);
                    todo.push_back(b);
                }
            }

            // The topology and every leaf's triangle SET are independent of the order in which subtrees are built
            // (a split only looks at its own range of `info`), so large scenes are built by a team of threads:
            // the top of the tree is opened sequentially until there are enough independent subtrees, these are
            // built into thread-private pools and spliced behind their roots. What the reference's single recursion
            // fixes beyond the topology -- the order in which leaves hand their triangles to the ordered array -- is
            // replayed afterwards by emitOrder().
            int build(unsigned int nTris, unsigned int threads)
            {
                pool.reserve(2 * (size_t)nTris);
                pool.push_back(BuildNode());
                std::vector<Task> frontier;
                frontier.push_back(Task{ 0, 0u, nTris });
                const size_t wanted = threads > 1 && nTris >= (1u << 16) ? (size_t)threads * 8 : 1;
                while (frontier.size() < wanted)
                {
                    // open the largest pending range
                    size_t big = 0;
                    for (size_t i = 1; i < frontier.size(); ++i)
                        if (frontier[i].end - frontier[i].start > frontier[big].end - frontier[big].start) big = i;
                    if (frontier[big].end - frontier[big].start < 4096) break;
                    Task t = frontier[big], a, b;
                    frontier.erase(frontier.begin() + big);
                    if (expand(pool, t, a, b)) { frontier.push_back(a); frontier.push_back(b); }
                    if (frontier.empty()) break;
                }
                if (wanted == 1 || frontier.size() < 2)
                {
                    for (const Task& t : frontier) buildSubtree(pool, t);
                }
                else
                {
                    std::sort(frontier.begin(), frontier.end(), [](const Task& x, const Task& y) { return x.end - x.start > y.end - y.start; });
                    std::vector<std::vector<BuildNode>> local(frontier.size());
                    std::atomic<size_t> next(0);
                    auto work = [&]() {
                        for (size_t i = next.fetch_add(1); i < frontier.size(); i = next.fetch_add(1))
                        {
                            local[i].reserve(2 * (size_t)(frontier[i].end - frontier[i].start));
                            local[i].push_back(BuildNode());
                            buildSubtree(local[i], Task{ 0, frontier[i].start, frontier[i].end });
                        }
                    };
                    std::vector<std::thread> team;
                    for (unsigned int k = 1; k < threads; ++k) team.emplace_back(work);
                    work();
                    for (std::thread& th : team) th.join();
                    // splice: local node 0 becomes the frontier node, local node j > 0 becomes pool[base + j - 1]
                    for (size_t i = 0; i < frontier.size(); ++i)
                    {
                        const int base = (int)pool.size();
                        auto remap = [&](BuildNode n) { if (n.child[0] >= 0) { n.child[0] += base - 1; n.child[1] += base - 1; } return n; };
                        pool[frontier[i].id] = remap(local[i][0]);
                        for (size_t j = 1; j < local[i].size(); ++j) pool.push_back(remap(local[i][j]));
                        std::vector<BuildNode>().swap(local[i]);
                    }
                }
                // interior bounds = union of the children, bottom-up (children always have larger pool ids)
                for (size_t i = pool.size(); i-- > 0;)
                    if (pool[i].child[0] >= 0) pool[i].bounds = Union(pool[pool[i].child[0]].bounds, pool[pool[i].child[1]].bounds);
                emitOrder(nTris);
                return 0;
            }

            // The reference appends a leaf's triangles to the ordered array when its recursion reaches that leaf, and
            // it recurses into the SECOND child first (see the header): replay exactly that walk.
            void emitOrder(unsigned int nTris)
            {
                order.clear();
                order.reserve(nTris);
                std::vector<int> todo;
                todo.push_back(0);
                while (!todo.empty())
                {
                    BuildNode& n = pool[todo.back()];
                    todo.pop_back();
                    if (n.child[0] < 0)
                    {
                        const unsigned int start = n.firstPrim;
                        n.firstPrim = (unsigned int)order.size();
                        for (unsigned int i = start; i < start + n.nPrims; ++i) order.push_back(info[i].prim);
                    }
                    else { todo.push_back(n.child[0]); todo.push_back(n.child[1]); }   // LIFO: second child first
                }
            }
        };
    }

    void CLBVHScene::BuildOnly(unsigned int maxPrimitivesInNode)
    {
        m_MaxPrimitivesInNode = maxPrimitivesInNode;
        m_Nodes.clear();
        if (m_Triangles.empty()) throw CLException("Cannot build a BVH over an empty scene", B2RT_INVALID_VALUE);
        if (m_Triangles.size() >= 0xfffffffeull) throw CLException("Scene too large", B2RT_INVALID_VALUE);
        Builder b;
        b.maxPrims = maxPrimitivesInNode;
        b.info.resize(m_Triangles.size());
        for (unsigned int i = 0; i < m_Triangles.size(); ++i)
        {
            CLBounds3 tb = m_Triangles[i].GetBounds();
            b.info[i] = PrimInfo{ i, tb, tb.min * 0.5f + tb.max * 0.5f };
        }
        unsigned int threads = std::thread::hardware_concurrency();
        if (const char* env = std::getenv("B2RT_BUILD_THREADS")) threads = (unsigned int)std::max(1, std::atoi(env));
        b.build((unsigned int)m_Triangles.size(), std::max(1u, std::min(threads, 64u)));
        std::vector<PrimInfo>().swap(b.info);

        // re-order the triangles
        {
            std::vector<CLTriangle> ordered;
            ordered.reserve(b.order.size());
            for (unsigned int src : b.order) ordered.push_back(m_Triangles[src]);
            m_Triangles.swap(ordered);
        }
        // pre-order numbering, first child at index + 1
        m_Nodes.resize(b.pool.size());
        struct Visit { int pool; int parent; };     // parent: linear index whose `offset` must point at this node, or -1
        std::vector<Visit> stack;
        stack.push_back(Visit{ 0, -1 });
        unsigned int next = 0;
        while (!stack.empty())
        {
            Visit v = stack.back();
            stack.pop_back();
            const BuildNode& n = b.pool[v.pool];
            unsigned int me = next++;
            if (v.parent >= 0) m_Nodes[v.parent].offset = me;
            CLLinearBVHNode& out = m_Nodes[me];
            out.bounds = n.bounds;
            if (n.child[0] < 0)
            {
                if (n.nPrims >= 65536) throw CLException("Leaf with more than 65535 primitives", B2RT_INVALID_VALUE);
                out.offset = n.firstPrim;
                out.nPrimitives = (unsigned short)n.nPrims;
            }
            else
            {
                out.axis = (unsigned char)n.axis;
                out.nPrimitives = 0;
                stack.push_back(Visit{ n.child[1], (int)me });   // numbered after the whole first subtree
                stack.push_back(Visit{ n.child[0], -1 });        // numbered next: index me + 1
            }
        }
        assert(next == m_Nodes.size());
    }

    void CLBVHScene::CreateBVHTrees(unsigned int maxPrimitivesInNode)
    {
        BuildOnly(maxPrimitivesInNode);
        if (eng && eng->render && eng->render->m_CLContext) SetupBuffers();
    }

    void CLBVHScene::CreateBVHTreesDevice()
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::CreateBVHTreesDevice needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        if (m_Triangles.empty()) throw CLException("Cannot build a BVH over an empty scene", B2RT_INVALID_VALUE);
        b2rt_context* ctx = eng->render->m_CLContext->GetContext();
        std::vector<CLLinearBVHNode> nodes(2 * m_Triangles.size() - 1);
        std::vector<uint32_t> order(m_Triangles.size());
        uint64_t n_nodes = 0;
        int st = b2rt_build_bvh(ctx, m_Triangles.data(), m_Triangles.size(), nodes.data(), nodes.size(), &n_nodes, order.data());
        if (st) throw CLException(std::string("Failed to build the BVH on the device: ") + b2rt_last_error(ctx), st);
        nodes.resize(n_nodes);
        // re-order m_Triangles like CreateBVHTrees does (CLBVHnode.cpp:197): a 256-byte gather per triangle, split over a team
        std::vector<CLTriangle> ordered(order.size());
        const size_t n = order.size();
        const unsigned team = (unsigned)std::max<size_t>(1, std::min<size_t>({ (size_t)std::thread::hardware_concurrency(), n / 65536 + 1, 16 }));
        auto gather = [&](size_t lo, size_t hi) { for (size_t k = lo; k < hi; ++k) ordered[k] = m_Triangles[order[k]]; };
        if (team <= 1) gather(0, n);
        else {
            std::vector<std::thread> pool;
            for (unsigned w = 0; w < team; ++w) pool.emplace_back(gather, n * w / team, n * (w + 1) / team);
            for (auto& t : pool) t.join();
        }
        m_Triangles.swap(ordered);
        m_Nodes.swap(nodes);
        SetupBuffers();
    }

    void CLBVHScene::CreateBVHTreesFromDevice(const void* d_triangles, size_t n)
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::CreateBVHTreesFromDevice needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        if (m_Materials.empty()) throw CLException("CLBVHScene::CreateBVHTreesFromDevice needs the scene's materials", B2RT_INVALID_VALUE);
        const CLContext& ctx = *eng->render->m_CLContext;
        b2rt_context* c = ctx.GetContext();
        int err = 0;
        m_MaterialBuffer = CLBuffer(ctx, B2RT_MEM_READ_ONLY | B2RT_MEM_COPY_HOST_PTR, m_Materials.size() * sizeof(CLMaterial), m_Materials.data(), &err);
        if (err) throw CLException("Failed to create material buffer", err);
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_MATERIAL, m_MaterialBuffer);
        CLBuffer order(ctx, 0, n * sizeof(uint32_t), nullptr, &err);
        if (err) throw CLException("Failed to create triangle order buffer", err);
        void* d_order = nullptr;
        err = b2rt_device_pointer(c, order.id(), &d_order, nullptr);
        if (err) throw CLException("Failed to find the triangle order buffer", err);
        b2rt_buffer bt = 0, bn = 0;
        uint64_t n_nodes = 0;
        int st = b2rt_build_scene_device(c, d_triangles, n, static_cast<uint32_t*>(d_order), &bt, &bn, &n_nodes, nullptr);
        if (st) throw CLException(std::string("Failed to build the scene on the device: ") + b2rt_last_error(c), st);
        m_OrderBuffer = order;
        // the library has bound both buffers already; binding the same ids again changes nothing
        m_TriangleBuffer = CLBuffer::Adopt(ctx, bt, n * sizeof(CLTriangle));
        m_NodeBuffer = CLBuffer::Adopt(ctx, bn, (size_t)n_nodes * sizeof(CLLinearBVHNode));
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_SCENE, m_TriangleBuffer);
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_NODE, m_NodeBuffer);
        m_Triangles.clear();
        m_Nodes.clear();
    }

    void CLBVHScene::ReadBackScene()
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::ReadBackScene needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        if (!m_TriangleBuffer.id() || !m_NodeBuffer.id()) throw CLException("CLBVHScene::ReadBackScene needs a scene on the device", B2RT_INVALID_MEM_OBJECT);
        b2rt_context* c = eng->render->m_CLContext->GetContext();
        m_Triangles.resize(m_TriangleBuffer.size() / sizeof(CLTriangle));
        m_Nodes.resize(m_NodeBuffer.size() / sizeof(CLLinearBVHNode));
        int st = b2rt_read_buffer(c, m_TriangleBuffer.id(), m_Triangles.data(), m_Triangles.size() * sizeof(CLTriangle));
        if (!st) st = b2rt_read_buffer(c, m_NodeBuffer.id(), m_Nodes.data(), m_Nodes.size() * sizeof(CLLinearBVHNode));
        if (!st) st = b2rt_finish(c);
        if (st) throw CLException(std::string("Failed to read the scene back: ") + b2rt_last_error(c), st);
    }

    void CLBVHScene::SetupBuffers()
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::SetupBuffers needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        const CLContext& ctx = *eng->render->m_CLContext;
        int err = 0;
        m_TriangleBuffer = CLBuffer(ctx, B2RT_MEM_READ_ONLY | B2RT_MEM_COPY_HOST_PTR, m_Triangles.size() * sizeof(CLTriangle), m_Triangles.data(), &err);
        if (err) throw CLException("Failed to create scene buffer", err);
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_SCENE, m_TriangleBuffer);
        m_NodeBuffer = CLBuffer(ctx, B2RT_MEM_READ_ONLY | B2RT_MEM_COPY_HOST_PTR, m_Nodes.size() * sizeof(CLLinearBVHNode), m_Nodes.data(), &err);
        if (err) throw CLException("Failed to create BVH node buffer", err);
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_NODE, m_NodeBuffer);
        m_MaterialBuffer = CLBuffer(ctx, B2RT_MEM_READ_ONLY | B2RT_MEM_COPY_HOST_PTR, m_Materials.size() * sizeof(CLMaterial), m_Materials.data(), &err);
        if (err) throw CLException("Failed to create material buffer", err);
        eng->render->SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_MATERIAL, m_MaterialBuffer);
        m_OrderBuffer = CLBuffer();                                    // the triangles uploaded here are in scene order
    }

    void CLBVHScene::Refit()
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::Refit needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        if (!m_TriangleBuffer.id() || !m_NodeBuffer.id()) throw CLException("CLBVHScene::Refit needs an uploaded scene", B2RT_INVALID_MEM_OBJECT);
        b2rt_context* c = eng->render->m_CLContext->GetContext();
        int st = b2rt_refit_scene(c, m_Triangles.data(), m_Triangles.size());
        if (st) throw CLException(std::string("Failed to refit scene: ") + b2rt_last_error(c), st);
        st = b2rt_read_buffer(c, m_NodeBuffer.id(), m_Nodes.data(), m_Nodes.size() * sizeof(CLLinearBVHNode));
        if (!st) st = b2rt_finish(c);
        if (st) throw CLException(std::string("Failed to read refitted nodes: ") + b2rt_last_error(c), st);
    }

    void CLBVHScene::RefitFromDevice(const void* d_triangles, size_t n)
    {
        if (!eng || !eng->render || !eng->render->m_CLContext)
            throw CLException("CLBVHScene::RefitFromDevice needs eng->render->m_CLContext", B2RT_INVALID_CONTEXT);
        if (!m_TriangleBuffer.id() || !m_NodeBuffer.id()) throw CLException("CLBVHScene::RefitFromDevice needs a scene on the device", B2RT_INVALID_MEM_OBJECT);
        const CLContext& ctx = *eng->render->m_CLContext;
        b2rt_context* c = ctx.GetContext();
        int err = 0;
        if (!m_RefitStatusBuffer.id()) {
            m_RefitStatusBuffer = CLBuffer(ctx, 0, sizeof(uint32_t), nullptr, &err);
            if (err) throw CLException("Failed to create refit status buffer", err);
        }
        const CLBuffer& status = m_RefitStatusBuffer;
        void *d_status = nullptr, *d_order = nullptr;
        err = b2rt_device_pointer(c, status.id(), &d_status, nullptr);
        if (!err && m_OrderBuffer.id()) err = b2rt_device_pointer(c, m_OrderBuffer.id(), &d_order, nullptr);
        if (err) throw CLException("Failed to find the refit buffers", err);
        int st = b2rt_refit_scene_device(c, d_triangles, n, static_cast<const uint32_t*>(d_order), static_cast<uint32_t*>(d_status), nullptr);
        if (st) throw CLException(std::string("Failed to refit scene: ") + b2rt_last_error(c), st);
        uint32_t bits = 0;
        st = b2rt_read_buffer(c, status.id(), &bits, sizeof(bits));
        if (!st) st = b2rt_finish(c);
        if (st) throw CLException(std::string("Failed to read the refit status: ") + b2rt_last_error(c), st);
        if (bits) {
            static const char* names[] = { "non-finite vertex positions", "a loader duplicate pair was broken (rebuild instead)",
                                           "bounds too large to quantise", "a leaf box no longer matches its vertices",
                                           "a triangle order entry out of range" };
            std::string what;
            for (int b = 0; b < 5; ++b)
                if (bits & (1u << b)) what += (what.empty() ? "" : "; ") + std::string(names[b]);
            throw CLException("Failed to refit scene: " + what, B2RT_INVALID_ARG_VALUE);
        }
    }
}
