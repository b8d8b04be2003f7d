// glaze3d.h -- headless C++ mirror of the reference's host-side API (namespace Glaze3D), re-pointed
// from OpenCL at the C ABI of libb2rt.so (include/b2rt.h). A program written against the reference's
// CLRaytracer / CLEngineBase / CLContext / CLKernel / CLBVHScene / CLOBJloader keeps compiling against
// this header; everything GUI (GLFW, GLEW, ImGui, WinMain, MessageBox) is gone.
//
// What is mirrored, with the reference location of each piece:
//   float3 / float2 / CLBounds3 .......... CLmathlib.hpp:18-204 (16-byte float3, Union, SurfaceArea, ...)
//   CLMaterial / CLVertex / CLTriangle /
//   CLLinearBVHNode ....................... CLshared_structs.hpp:13-88 (byte-identical: 64/80/256/48 B)
//   CLCamera / CLLight .................... CLcamera.h:6-21, CLLight.h:6-13
//   RenderKernelArgument_t, CLException,
//   GetClErrorString, CLContext, CLKernel . CLutils.h:11-145
//   CLBVHScene ............................ clBVHnode.h:52-79, CLBVHnode.cpp:7-236
//   CLOBJloader ........................... CLOBJloader.h, CLOBJloader.cpp:10-176
//   CLRaytracer ........................... CLRaytracer.h:16-40, CLRaytracer.cpp:12-148
//   CLui (state only) / CLEngineBase ...... CLui.h:17-40, CLEngineBase.h:13-93, CLEngineBase.cpp:141-211
// New (the reference has no ray-stream API): CLRaytracer::TraceClosest / TraceAny / TraceMulti / ClosestPoint / TraceRadiance.
#pragma once
#include <cstddef>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#include "b2rt.h"

namespace Glaze3D
{
    // ---- math ---------------------------------------------------------------------------------
    struct vec3 { float x = 0, y = 0, z = 0; vec3() {} vec3(float a, float b, float c) : x(a), y(b), z(c) {} };   // stands in for glm::vec3

    class float3
    {
    public:
        float3() : x(0), y(0), z(0), w(0) {}
        float3(float v) : x(v), y(v), z(v), w(0) {}
        float3(float a, float b, float c) : x(a), y(b), z(c), w(0) {}
        float3(const vec3& v) : x(v.x), y(v.y), z(v.z), w(0) {}
        float& operator[](size_t i) { return i == 0 ? x : (i == 1 ? y : z); }
        const float& operator[](size_t i) const { return i == 0 ? x : (i == 1 ? y : z); }
        float x, y, z;
    private:
        float w;   // pads the struct to the 16 bytes an OpenCL float3 occupies (the reference leaves it uninitialised)
    };
    static_assert(sizeof(float3) == 16, "float3 must be 16 bytes (CLmathlib.hpp:18-54)");
    inline float3 operator+(const float3& a, const float3& b) { return float3(a.x + b.x, a.y + b.y, a.z + b.z); }
    inline float3 operator-(const float3& a, const float3& b) { return float3(a.x - b.x, a.y - b.y, a.z - b.z); }
    inline float3 operator*(const float3& a, float s) { return float3(a.x * s, a.y * s, a.z * s); }

    struct float2 { float x = 0, y = 0; float2() {} float2(float a, float b) : x(a), y(b) {} };

    struct CLBounds3
    {
        CLBounds3();                                  // empty: min = +FLT_MAX, max = -FLT_MAX
        CLBounds3(const float3& p) : min(p), max(p) {}
        CLBounds3(const float3& a, const float3& b);
        float3 Diagonal() const { return max - min; }
        float SurfaceArea() const { float3 d = Diagonal(); return 2 * (d.x * d.y + d.x * d.z + d.y * d.z); }
        unsigned int MaximumExtent() const;
        float3 Offset(const float3& p) const;
        float3 min, max;
    };
    CLBounds3 Union(const CLBounds3& b, const float3& p);
    CLBounds3 Union(const CLBounds3& a, const CLBounds3& b);

    // ---- device-shared PODs (CLshared_structs.hpp) -----------------------------------------------
    struct CLMaterial
    {
        CLMaterial() : diffuse(0.2f), specular(1.0f), emission(0.0f), type(0), roughness(9999.0f), ior(0.0f), padding(0) {}
        float3 diffuse, specular, emission;
        unsigned int type;
        float roughness, ior;
        int padding;
    };
    struct CLVertex
    {
        CLVertex() {}
        CLVertex(const float3& p, const float2& t, const float3& n) : position(p), uv(t.x, t.y, 0), normal(n) {}
        float3 position, uv, normal, tangent_s, tangent_t;
    };
    struct CLTriangle
    {
        CLTriangle() : mtlIndex(0), padding{ 0, 0, 0 } {}
        CLTriangle(const CLVertex& a, const CLVertex& b, const CLVertex& c, unsigned int m) : v1(a), v2(b), v3(c), mtlIndex(m), padding{ 0, 0, 0 } {}
        CLBounds3 GetBounds() const { return Union(CLBounds3(v1.position, v2.position), v3.position); }
        CLVertex v1, v2, v3;
        unsigned int mtlIndex;
        unsigned int padding[3];
    };
    struct CLLinearBVHNode
    {
        CLLinearBVHNode() : offset(0), nPrimitives(0), axis(0), pad{ 0 } {}
        CLBounds3 bounds;
        unsigned int offset;          // leaf: first triangle; interior: index of the second child (first child = this + 1)
        unsigned short nPrimitives;   // 0 -> interior
        unsigned char axis;           // interior: split axis
        unsigned char pad[9];
    };
    static_assert(sizeof(CLMaterial) == 64 && sizeof(CLVertex) == 80 && sizeof(CLTriangle) == 256 && sizeof(CLLinearBVHNode) == 48,
                  "device-shared layouts must match CLshared_structs.hpp byte for byte");

    // ---- camera / light ------------------------------------------------------------------------
    struct CLCamera
    {
        vec3 position = vec3(0.0f, -25.0f, 8.5f);
        vec3 front = vec3(0.0f, 1.0f, 0.0f);
        vec3 up = vec3(0.0f, 0.0f, 1.0f);
        vec3 right = vec3(1.0f, 0.0f, 0.0f);
        float pitch = 1.571f;
        float yaw = 1.571f;
        void Update();
    };
    struct CLLight   // never sent to the kernel by the reference either (kernel_bvh.cl:307-309 hard-codes its own)
    {
        vec3 position = vec3(0.0f, -10.0f, 16.0f);
        vec3 direction = vec3(-0.5f, 0.4f, -0.1f);
        int type = 0;
        float intensity = 1.0f;
        float attenuation = 0.6f;
    };

    // ---- device runtime wrapper (CLutils.h) -------------------------------------------------------
    enum class RenderKernelArgument_t : unsigned int
    {
        BUFFER_OUT, BUFFER_SCENE, BUFFER_NODE, BUFFER_MATERIAL, WIDTH, HEIGHT, FRAME_COUNT, FRAME_SEED,
        LIGHT_BOUNCES, LIGHT_TYPE, SKYBOX_INTENSITY, CAMERA_POS, CAMERA_FRONT, CAMERA_UP
    };
    inline const char* GetClErrorString(int error) { return b2rt_status_string(error); }

    class CLException : public std::runtime_error
    {
    public:
        CLException(const std::string& message, int errorCode)
            : std::runtime_error(message + " (" + GetClErrorString(errorCode) + ")"), code(errorCode) {}
        int code;
    };

    class CLContext;
    // Stands in for cl::Buffer: a shared handle to a device allocation owned by a CLContext.
    class CLBuffer
    {
    public:
        CLBuffer() {}
        // cl::Buffer(context, flags, size, host_ptr, &err)
        CLBuffer(const CLContext& context, uint32_t flags, size_t size, const void* host_ptr, int* err);
        // New: take ownership of a buffer the library created (e.g. by b2rt_build_scene_device); released like any other
        static CLBuffer Adopt(const CLContext& context, b2rt_buffer id, size_t size);
        b2rt_buffer id() const { return m_State ? m_State->id : 0; }
        size_t size() const { return m_State ? m_State->bytes : 0; }
    private:
        struct State { b2rt_context* ctx; b2rt_buffer id; size_t bytes; ~State(); };
        std::shared_ptr<State> m_State;
    };

    class CLKernel;
    class CLContext
    {
    public:
        explicit CLContext(int device = 0);            // the reference takes a cl::Platform and uses its device 0
        // All of these devices behind one context (b2rt_create_multi): what the reference's context over
        // platform.getDevices(CL_DEVICE_TYPE_ALL) (CLutils.cpp:20-26) promises and its single queue never delivers.
        explicit CLContext(const std::vector<int>& devices);
        ~CLContext();
        CLContext(const CLContext&) = delete;
        CLContext& operator=(const CLContext&) = delete;
        void ReadBuffer(const CLBuffer& buffer, void* ptr, size_t size) const;      // non-blocking, like CLutils.cpp:37-42
        void ExecuteKernel(std::shared_ptr<CLKernel> kernel, size_t workSize) const;
        void ExecuteKernelRange(std::shared_ptr<CLKernel> kernel, size_t gidBegin, size_t gidEnd) const;   // one screen shard
        void Finish() const;
        b2rt_context* GetContext() const { return m_Context; }
        int Device() const { return m_Device; }
    private:
        b2rt_context* m_Context = nullptr;
        int m_Device = 0;
    };

    class CLKernel
    {
    public:
        // The reference JIT-compiles `filename` (kernel_bvh.cl) here; this build ships precompiled sm_100a
        // kernels inside libb2rt.so, so the name is only recorded.
        CLKernel(const char* filename, const CLContext& context);
        bool SetArgument(RenderKernelArgument_t argIndex, void* data, size_t size);
        const std::string& Name() const { return m_File; }
    private:
        b2rt_context* m_Context;
        std::string m_File;
    };

    // ---- scene ----------------------------------------------------------------------------------
    class CLBVHScene
    {
    public:
        std::vector<CLTriangle> m_Triangles;
        std::vector<CLMaterial> m_Materials;
        std::vector<std::string> m_MaterialNames;
        unsigned int m_MaxPrimitivesInNode = 0;

        CLBVHScene() {}
        // Builds the SAH BVH over m_Triangles (re-ordering them), flattens it and, when an engine with a
        // renderer exists (`eng->render`), uploads the three arrays like the reference does.
        void CreateBVHTrees(unsigned int maxPrimitivesInNode);
        void BuildOnly(unsigned int maxPrimitivesInNode);                 // build + flatten, no upload
        // Same result TYPE as CreateBVHTrees (re-ordered m_Triangles + flattened node array, uploaded), but the tree is
        // built on the GPU by b2rt_build_bvh (Morton order + Karras hierarchy) instead of the SAH recursion: a few
        // milliseconds of device time instead of seconds. It is a different tree: hit IDs index THIS order.
        void CreateBVHTreesDevice();
        // New: the whole scene built on the GPU from n LOADER-order triangles already in device memory of the context's
        // device (b2rt_build_scene_device): m_Materials are uploaded and bound first, then the tree, the re-ordered
        // triangles and the compressed wide BVH are made on the device. The re-ordered triangles and the node array stay
        // there, held by m_TriangleBuffer / m_NodeBuffer; m_Triangles and Nodes() stay empty until ReadBackScene(). The
        // triangle order of the build stays on the device too (m_OrderBuffer), for RefitFromDevice.
        void CreateBVHTreesFromDevice(const void* d_triangles, size_t n);
        void ReadBackScene();                                             // m_TriangleBuffer / m_NodeBuffer -> m_Triangles / Nodes()
        // New: the vertices of m_Triangles were changed in place (same count and order): refit the device scene -- node boxes,
        // compressed wide BVH, shading records -- by b2rt_refit_scene instead of building and uploading again, and read the
        // refitted node boxes back into Nodes().
        void Refit();
        // New: refit the device scene from n triangles already in device memory of the context's device
        // (b2rt_refit_scene_device): in LOADER order for a scene made by CreateBVHTreesFromDevice (gathered through
        // m_OrderBuffer), in scene order for a scene built or uploaded from the host. Synchronous; a status bit set by the
        // refit throws CLException(B2RT_INVALID_ARG_VALUE) naming it. m_Triangles / Nodes() are left as they are (stale);
        // ReadBackScene() refreshes them.
        void RefitFromDevice(const void* d_triangles, size_t n);
        const std::vector<CLLinearBVHNode>& Nodes() const { return m_Nodes; }
        void SetupBuffers();                                              // CLBVHnode.cpp:209-236

        // Binary cache of the post-loader, post-build arrays (scene_cache.cpp): a hit restores m_Triangles (in their
        // post-build order, i.e. identical hit IDs), the node array, materials and names without parsing or building.
        static std::string CachePathFor(const char* objPath, unsigned int maxPrimitivesInNode);
        void SaveCache(const char* cachePath, const char* objPath) const;
        bool LoadCache(const char* cachePath, const char* objPath, unsigned int maxPrimitivesInNode);   // false = missing / stale / corrupt
    private:
        std::vector<CLLinearBVHNode> m_Nodes;
        CLBuffer m_TriangleBuffer, m_NodeBuffer, m_MaterialBuffer;
        CLBuffer m_OrderBuffer;           // uint32 per triangle: loader index of scene triangle k (device-built scenes only)
        CLBuffer m_RefitStatusBuffer;     // uint32: RefitFromDevice's status word, made on its first call
    };

    class CLOBJloader
    {
    public:
        CLOBJloader() {}
        void Load(const char* filename, unsigned int maxPrimitivesInNode);            // into eng->render->m_Scene
        static void LoadInto(CLBVHScene& scene, const char* filename);                 // same parser, explicit target
        // Load + build through the binary cache (cachePath null/empty = beside the .obj). Returns true on a cache hit;
        // on a miss the scene is parsed and built as usual and the cache is (re)written.
        static bool LoadCached(CLBVHScene& scene, const char* filename, unsigned int maxPrimitivesInNode, const char* cachePath = nullptr);
    };

    // ---- renderer -------------------------------------------------------------------------------
    class CLRaytracer
    {
    public:
        ~CLRaytracer();
        void Init();
        void RenderFrame();
        template <class T> bool SetUniform(int i, T& val);
        void SetupBuffers();

        // New: ray streams through the same scene. hits[i].tri == B2RT_MISS on a miss.
        void TraceClosest(const b2rt_ray* rays, uint64_t n, b2rt_hit* hits);
        void TraceAny(const b2rt_ray* rays, uint64_t n, uint32_t* occluded);
        // The k nearest hits per ray (b2rt_trace_multi): hits[i*k .. i*k+k) sorted by t, unused slots {tmax, 0, 0, B2RT_MISS}.
        void TraceMulti(const b2rt_ray* rays, uint64_t n, uint32_t k, b2rt_hit* hits);
        // The nearest surface point per query point (b2rt_closest_point): out[i] = {d2, u, v, tri}, {max_d2, 0, 0, B2RT_MISS} if none.
        void ClosestPoint(const b2rt_point_query* queries, uint64_t n, b2rt_point_hit* out);
        // The path-traced radiance per ray (b2rt_trace_radiance): out[i] = {r, g, b, RNG state after the path}, shaded with
        // the bound light bounces, light type, sky intensity and materials.
        void TraceRadiance(const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out);

        std::shared_ptr<CLContext> m_CLContext = nullptr;
        std::shared_ptr<CLKernel> m_RenderKernel = nullptr;
        std::shared_ptr<CLBVHScene> m_Scene = nullptr;

        unsigned int m_FrameCount = 1;
        int lightType = 0;
        int lightBounces = 9;
        int dofOn = 0;
        float skyboxIntensity = 1.0f;

        std::vector<float3> pixels;
        // Display read-back (new): when set, RenderFrame fetches the frame as clamped 8-bit RGBA quantised on the device
        // (4 B/pixel) into pixels8 instead of the 16 B/pixel float image into `pixels` -- what the reference's
        // glTexImage2D(GL_RGBA, GL_FLOAT) upload of `pixels` displays (CLRaytracer.cpp:64-67).
        bool displayReadback = false;
        std::vector<uint32_t> pixels8;
        CLBuffer m_OutputBuffer;
        int device = 0;                 // which GPU Init() opens
        std::vector<int> devices;       // non-empty: Init() opens ALL of these behind one context; RenderFrame then splits every
                                        // frame into screen bands over them and reads the gathered image from devices[0]
        size_t shardBegin = 0, shardEnd = 0;   // [begin,end) of gids this renderer draws; 0,0 = whole frame
    };

    template <> bool CLRaytracer::SetUniform<CLBuffer>(int i, CLBuffer& val);     // passes the buffer handle (runtime.cpp)

    // Window / UI state the render path reads (CLui.h:17-40). No window is ever created.
    class CLui
    {
    public:
        int window_width = 1280, window_height = 720;
        bool isPaused = false, framestepOn = false, windowClose = false, firstRun = true;
    };

    class CLEngineBase
    {
    public:
        CLEngineBase();
        void init();                                    // headless: nothing to open
        void processInput() {}                          // no keyboard
        // CLEngineBase::renderLoop (CLEngineBase.cpp:166-211) without the window: Init, load `scene`
        // (the reference hard-codes "cornell.obj", maxPrimitives 4), render `frames` frames.
        void renderLoop(const std::string& scene = "cornell.obj", unsigned int frames = 1, unsigned int maxPrimitives = 4);

        bool isInitialized = false;
        bool windowClose = false;
        bool sceneCache = false;                        // renderLoop loads scenes through CLOBJloader::LoadCached
        float FPS = 0;
        std::shared_ptr<CLRaytracer> render = nullptr;
        std::shared_ptr<CLui> ui = nullptr;
        CLCamera m_Camera;
        CLLight m_Light;
    };

    extern std::shared_ptr<CLEngineBase> eng;          // the reference's global singleton (stdafx.h:106-110, main.cpp:5)
}
