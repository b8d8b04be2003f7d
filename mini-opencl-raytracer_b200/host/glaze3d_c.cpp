// glaze3d_c.cpp -- flat C view of the C++ host mirror (glaze3d.h) for harnesses that cannot link C++
// (bench.py / the tests bind it with ctypes). Exceptions never cross this boundary: every call returns
// 0 / a handle on success and copies the CLException text into the caller's buffer on failure.
#include <cstdio>
#include <cstring>
#include "glaze3d.h"

using namespace Glaze3D;

namespace
{
    void setError(char* err, size_t errLen, const char* text)
    {
        if (err && errLen) { std::snprintf(err, errLen, "%s", text); }
    }
    struct SceneBox { std::shared_ptr<CLBVHScene> scene; };
    struct EngineBox { std::shared_ptr<CLEngineBase> engine; };
}

#define G3D_TRY try {
#define G3D_CATCH(failValue)                                                                  \
    } catch (const std::exception& e) { setError(err, errLen, e.what()); return failValue; } \
      catch (...) { setError(err, errLen, "unknown exception"); return failValue; }


// ---- scenes without a device: CLOBJloader + CLBVHScene::BuildOnly ---------------------------------
extern "C" void* g3d_scene_load(const char* objPath, unsigned maxPrims, char* err, size_t errLen)
{
    G3D_TRY
    auto s = std::make_shared<CLBVHScene>();
    s->m_MaxPrimitivesInNode = maxPrims;
    CLOBJloader::LoadInto(*s, objPath);
    s->BuildOnly(maxPrims);
    return new SceneBox{ s };
    G3D_CATCH(nullptr)
}
// Same through the binary scene cache; *hit (optional) reports whether the cache was used.
extern "C" void* g3d_scene_load_cached(const char* objPath, unsigned maxPrims, const char* cachePath, int* hit, char* err, size_t errLen)
{
    G3D_TRY
    auto s = std::make_shared<CLBVHScene>();
    bool h = CLOBJloader::LoadCached(*s, objPath, maxPrims, cachePath);
    if (hit) *hit = h ? 1 : 0;
    return new SceneBox{ s };
    G3D_CATCH(nullptr)
}
// CLOBJloader only: the triangles in LOADER order, no BVH (input of b2rt_build_bvh).
extern "C" void* g3d_scene_load_triangles(const char* objPath, char* err, size_t errLen)
{
    G3D_TRY
    auto s = std::make_shared<CLBVHScene>();
    CLOBJloader::LoadInto(*s, objPath);
    return new SceneBox{ s };
    G3D_CATCH(nullptr)
}
extern "C" void* g3d_scene_from_triangles(const void* tris, uint64_t nTris, const void* mats, uint64_t nMats, unsigned maxPrims, char* err, size_t errLen)
{
    G3D_TRY
    auto s = std::make_shared<CLBVHScene>();
    const CLTriangle* t = static_cast<const CLTriangle*>(tris);
    s->m_Triangles.assign(t, t + nTris);
    const CLMaterial* m = static_cast<const CLMaterial*>(mats);
    s->m_Materials.assign(m, m + nMats);
    s->BuildOnly(maxPrims);
    return new SceneBox{ s };
    G3D_CATCH(nullptr)
}
extern "C" void g3d_scene_free(void* scene) { delete static_cast<SceneBox*>(scene); }
// which: 0 triangles (256 B), 1 nodes (48 B), 2 materials (64 B)
extern "C" uint64_t g3d_scene_count(void* scene, int which)
{
    CLBVHScene& s = *static_cast<SceneBox*>(scene)->scene;
    return which == 0 ? s.m_Triangles.size() : (which == 1 ? s.Nodes().size() : s.m_Materials.size());
}
extern "C" const void* g3d_scene_data(void* scene, int which)
{
    CLBVHScene& s = *static_cast<SceneBox*>(scene)->scene;
    return which == 0 ? (const void*)s.m_Triangles.data() : (which == 1 ? (const void*)s.Nodes().data() : (const void*)s.m_Materials.data());
}

// ---- the engine: CLEngineBase + CLRaytracer on one GPU (the reference's global `eng`) ----------------
extern "C" void* g3d_engine_create(int device, int width, int height, char* err, size_t errLen)
{
    G3D_TRY
    auto e = std::make_shared<CLEngineBase>();
    e->ui->window_width = width;
    e->ui->window_height = height;
    e->render->device = device;
    eng = e;
    e->init();
    e->render->Init();
    return new EngineBox{ e };
    G3D_CATCH(nullptr)
}
extern "C" void g3d_engine_destroy(void* engine)
{
    EngineBox* b = static_cast<EngineBox*>(engine);
    if (!b) return;
    if (eng == b->engine) eng.reset();
    delete b;
}
// CLEngineBase.cpp:172-179: new scene, CLOBJloader::Load, CreateBVHTrees (which uploads).
extern "C" int g3d_engine_load_scene(void* engine, const char* objPath, unsigned maxPrims, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->m_Scene = std::make_shared<CLBVHScene>();
    CLOBJloader loader;
    loader.Load(objPath, maxPrims);
    e->render->m_Scene->CreateBVHTrees(maxPrims);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_load_scene_cached(void* engine, const char* objPath, unsigned maxPrims, const char* cachePath, int* hit, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->m_Scene = std::make_shared<CLBVHScene>();
    bool h = CLOBJloader::LoadCached(*e->render->m_Scene, objPath, maxPrims, cachePath);
    if (hit) *hit = h ? 1 : 0;
    e->render->m_Scene->SetupBuffers();
    return 0;
    G3D_CATCH(-1)
}
// CLOBJloader::Load, then the BVH built on the GPU (CLBVHScene::CreateBVHTreesDevice) instead of the SAH recursion.
extern "C" int g3d_engine_load_scene_device_bvh(void* engine, const char* objPath, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->m_Scene = std::make_shared<CLBVHScene>();
    CLOBJloader loader;
    loader.Load(objPath, 4);
    e->render->m_Scene->CreateBVHTreesDevice();
    return 0;
    G3D_CATCH(-1)
}
// A new scene whose triangles are already on the device: CLBVHScene::CreateBVHTreesFromDevice with these materials.
extern "C" int g3d_engine_scene_from_device(void* engine, const void* d_triangles, uint64_t n, const void* materials, uint64_t n_materials,
                                            char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    auto scene = std::make_shared<CLBVHScene>();
    const CLMaterial* m = static_cast<const CLMaterial*>(materials);
    scene->m_Materials.assign(m, m + n_materials);
    e->render->m_Scene = scene;
    scene->CreateBVHTreesFromDevice(d_triangles, (size_t)n);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_scene_read_back(void* engine, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->m_Scene->ReadBackScene();
    return 0;
    G3D_CATCH(-1)
}
// CLBVHScene::RefitFromDevice: new vertex data already on the device (loader order for a device-built scene). Returns the
// CLException's status (e.g. B2RT_INVALID_ARG_VALUE for a refit status bit), -1 for any other failure.
extern "C" int g3d_engine_scene_refit_device(void* engine, const void* d_triangles, uint64_t n, char* err, size_t errLen)
{
    try {
        auto& e = static_cast<EngineBox*>(engine)->engine;
        eng = e;
        e->render->m_Scene->RefitFromDevice(d_triangles, (size_t)n);
        return 0;
    } catch (const CLException& x) {
        setError(err, errLen, x.what());
        return x.code ? x.code : -1;
    } catch (const std::exception& x) {
        setError(err, errLen, x.what());
        return -1;
    } catch (...) {
        setError(err, errLen, "unknown exception");
        return -1;
    }
}
extern "C" int g3d_engine_adopt_scene(void* engine, void* scene, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->m_Scene = static_cast<SceneBox*>(scene)->scene;
    e->render->m_Scene->SetupBuffers();
    return 0;
    G3D_CATCH(-1)
}
extern "C" void g3d_engine_set_camera(void* engine, const float* pos, const float* front, const float* up)
{
    auto& e = static_cast<EngineBox*>(engine)->engine;
    e->m_Camera.position = vec3(pos[0], pos[1], pos[2]);
    e->m_Camera.front = vec3(front[0], front[1], front[2]);
    e->m_Camera.up = vec3(up[0], up[1], up[2]);
}
extern "C" void g3d_engine_set_render(void* engine, unsigned frameCount, int lightBounces, int lightType, float skyboxIntensity)
{
    auto& r = static_cast<EngineBox*>(engine)->engine->render;
    r->m_FrameCount = frameCount;
    r->lightBounces = lightBounces;
    r->lightType = lightType;
    r->skyboxIntensity = skyboxIntensity;
}
extern "C" void g3d_engine_set_shard(void* engine, uint64_t gidBegin, uint64_t gidEnd)
{
    auto& r = static_cast<EngineBox*>(engine)->engine->render;
    r->shardBegin = (size_t)gidBegin;
    r->shardEnd = (size_t)gidEnd;
}
extern "C" int g3d_engine_render_frame(void* engine, char* err, size_t errLen)
{
    G3D_TRY
    auto& e = static_cast<EngineBox*>(engine)->engine;
    eng = e;
    e->render->RenderFrame();
    return 0;
    G3D_CATCH(-1)
}
extern "C" const float* g3d_engine_pixels(void* engine) { return &static_cast<EngineBox*>(engine)->engine->render->pixels[0].x; }
extern "C" void g3d_engine_set_display_readback(void* engine, int on) { static_cast<EngineBox*>(engine)->engine->render->displayReadback = on != 0; }
extern "C" const uint32_t* g3d_engine_pixels8(void* engine) { return static_cast<EngineBox*>(engine)->engine->render->pixels8.data(); }
extern "C" unsigned g3d_engine_frame_count(void* engine) { return static_cast<EngineBox*>(engine)->engine->render->m_FrameCount; }
extern "C" void* g3d_engine_context(void* engine) { return static_cast<EngineBox*>(engine)->engine->render->m_CLContext->GetContext(); }
extern "C" void* g3d_engine_scene(void* engine)
{
    auto& s = static_cast<EngineBox*>(engine)->engine->render->m_Scene;
    return s ? new SceneBox{ s } : nullptr;
}
extern "C" int g3d_engine_trace_closest(void* engine, const b2rt_ray* rays, uint64_t n, b2rt_hit* hits, char* err, size_t errLen)
{
    G3D_TRY
    static_cast<EngineBox*>(engine)->engine->render->TraceClosest(rays, n, hits);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_trace_any(void* engine, const b2rt_ray* rays, uint64_t n, uint32_t* occluded, char* err, size_t errLen)
{
    G3D_TRY
    static_cast<EngineBox*>(engine)->engine->render->TraceAny(rays, n, occluded);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_trace_multi(void* engine, const b2rt_ray* rays, uint64_t n, uint32_t k, b2rt_hit* hits, char* err, size_t errLen)
{
    G3D_TRY
    static_cast<EngineBox*>(engine)->engine->render->TraceMulti(rays, n, k, hits);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_closest_point(void* engine, const b2rt_point_query* queries, uint64_t n, b2rt_point_hit* out, char* err, size_t errLen)
{
    G3D_TRY
    static_cast<EngineBox*>(engine)->engine->render->ClosestPoint(queries, n, out);
    return 0;
    G3D_CATCH(-1)
}
extern "C" int g3d_engine_trace_radiance(void* engine, const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out, char* err,
                                         size_t errLen)
{
    G3D_TRY
    static_cast<EngineBox*>(engine)->engine->render->TraceRadiance(rays, seeds, n, out);
    return 0;
    G3D_CATCH(-1)
}
