// runtime.cpp -- CLBuffer / CLContext / CLKernel (the reference's OpenCL wrapper layer, CLutils.cpp:9-77),
// CLRaytracer (CLRaytracer.cpp:12-148) and the headless CLEngineBase, all as thin calls into the C ABI
// of libb2rt.so. Every non-zero status becomes a CLException with the reference's message text.
#include <chrono>
#include <cstdlib>
#include "glaze3d.h"

namespace Glaze3D
{
    std::shared_ptr<CLEngineBase> eng;

    // ---- CLBuffer ---------------------------------------------------------------------------------
    CLBuffer::State::~State() { if (ctx && id) b2rt_buffer_release(ctx, id); }

    CLBuffer::CLBuffer(const CLContext& context, uint32_t flags, size_t size, const void* host_ptr, int* err)
    {
        b2rt_buffer id = 0;
        int st = b2rt_buffer_create(context.GetContext(), flags, size, host_ptr, &id);
        if (err) *err = st;
        if (st == B2RT_SUCCESS) m_State = std::shared_ptr<State>(new State{ context.GetContext(), id, size });
    }

    CLBuffer CLBuffer::Adopt(const CLContext& context, b2rt_buffer id, size_t size)
    {
        CLBuffer b;
        if (id) b.m_State = std::shared_ptr<State>(new State{ context.GetContext(), id, size });
        return b;
    }

    // ---- CLContext --------------------------------------------------------------------------------
    CLContext::CLContext(int device) : m_Device(device)
    {
        int st = b2rt_create(device, &m_Context);
        if (st) throw CLException(std::string("Failed to create context: ") + b2rt_last_error(nullptr), st);
    }
    CLContext::CLContext(const std::vector<int>& devices) : m_Device(devices.empty() ? 0 : devices[0])
    {
        int st = b2rt_create_multi(devices.data(), (int)devices.size(), &m_Context);
        if (st) throw CLException(std::string("Failed to create context: ") + b2rt_last_error(nullptr), st);
    }
    CLContext::~CLContext() { b2rt_destroy(m_Context); }

    void CLContext::ReadBuffer(const CLBuffer& buffer, void* ptr, size_t size) const
    {
        int st = b2rt_read_buffer(m_Context, buffer.id(), ptr, size);
        if (st) throw CLException("Failed to read buffer", st);
    }
    void CLContext::ExecuteKernel(std::shared_ptr<CLKernel>, size_t workSize) const
    {
        int st = b2rt_execute(m_Context, workSize);
        if (st) throw CLException(std::string("Failed to enqueue kernel: ") + b2rt_last_error(m_Context), st);
    }
    void CLContext::ExecuteKernelRange(std::shared_ptr<CLKernel>, size_t gidBegin, size_t gidEnd) const
    {
        int st = b2rt_execute_range(m_Context, gidBegin, gidEnd);
        if (st) throw CLException(std::string("Failed to enqueue kernel: ") + b2rt_last_error(m_Context), st);
    }
    void CLContext::Finish() const
    {
        int st = b2rt_finish(m_Context);
        if (st) throw CLException(std::string("Failed to finish queue: ") + b2rt_last_error(m_Context), st);
    }

    // ---- CLKernel ---------------------------------------------------------------------------------
    CLKernel::CLKernel(const char* filename, const CLContext& context) : m_Context(context.GetContext()), m_File(filename ? filename : "") {}

    bool CLKernel::SetArgument(RenderKernelArgument_t argIndex, void* data, size_t size)
    {
        int st = b2rt_set_arg(m_Context, static_cast<unsigned int>(argIndex), data, size);
        if (st) throw CLException(std::string("Failed to set kernel argument: ") + b2rt_last_error(m_Context), st);
        return true;
    }

    // ---- CLRaytracer --------------------------------------------------------------------------------
    template <class T> bool CLRaytracer::SetUniform(int i, T& val)
    {
        return m_RenderKernel->SetArgument((RenderKernelArgument_t)i, &val, sizeof(T));
    }
    template <> bool CLRaytracer::SetUniform<CLBuffer>(int i, CLBuffer& val)
    {
        b2rt_buffer id = val.id();     // a buffer argument is passed as its handle, like clSetKernelArg(sizeof(cl_mem), &mem)
        return m_RenderKernel->SetArgument((RenderKernelArgument_t)i, &id, sizeof(id));
    }
    template bool CLRaytracer::SetUniform<float>(int, float&);
    template bool CLRaytracer::SetUniform<float3>(int, float3&);
    template bool CLRaytracer::SetUniform<int>(int, int&);
    template bool CLRaytracer::SetUniform<unsigned int>(int, unsigned int&);

    CLRaytracer::~CLRaytracer()
    {
        if (m_CLContext && !pixels.empty()) b2rt_host_unregister(m_CLContext->GetContext(), pixels.data());
        if (m_CLContext && !pixels8.empty()) b2rt_host_unregister(m_CLContext->GetContext(), pixels8.data());
    }

    void CLRaytracer::Init()
    {
        m_CLContext = devices.empty() ? std::make_shared<CLContext>(device) : std::make_shared<CLContext>(devices);
        m_RenderKernel = std::make_shared<CLKernel>("kernel_bvh.cl", *m_CLContext);
        SetupBuffers();
    }

    void CLRaytracer::SetupBuffers()
    {
        if (!eng || !eng->ui) throw CLException("CLRaytracer::SetupBuffers needs eng->ui", B2RT_INVALID_CONTEXT);
        int w = eng->ui->window_width, h = eng->ui->window_height;
        SetUniform<int>((int)RenderKernelArgument_t::WIDTH, w);
        SetUniform<int>((int)RenderKernelArgument_t::HEIGHT, h);
        if (!pixels.empty()) b2rt_host_unregister(m_CLContext->GetContext(), pixels.data());
        pixels.resize((size_t)w * h);
        // page-lock the read-back target: RenderFrame copies the whole frame into it every frame
        b2rt_host_register(m_CLContext->GetContext(), pixels.data(), pixels.size() * sizeof(float3));
        if (!pixels8.empty()) b2rt_host_unregister(m_CLContext->GetContext(), pixels8.data());
        pixels8.assign((size_t)w * h, 0u);
        b2rt_host_register(m_CLContext->GetContext(), pixels8.data(), pixels8.size() * sizeof(uint32_t));
        int err = 0;
        // Zero-filled by the library: the reference never clears it although frame 1 reads it (kernel_bvh.cl:454).
        m_OutputBuffer = CLBuffer(*m_CLContext, B2RT_MEM_WRITE_ONLY, (size_t)w * h * sizeof(float3), nullptr, &err);
        if (err) throw CLException("Failed to create output buffer", err);
        SetUniform<CLBuffer>((int)RenderKernelArgument_t::BUFFER_OUT, m_OutputBuffer);
    }

    void CLRaytracer::RenderFrame()
    {
        if (eng->ui->windowClose) return;
        unsigned int seed = (unsigned int)std::rand();           // sent and ignored, like the reference's kernel does
        SetUniform<unsigned int>((int)RenderKernelArgument_t::FRAME_COUNT, m_FrameCount);
        SetUniform<unsigned int>((int)RenderKernelArgument_t::FRAME_SEED, seed);
        SetUniform<int>((int)RenderKernelArgument_t::LIGHT_BOUNCES, lightBounces);
        SetUniform<int>((int)RenderKernelArgument_t::LIGHT_TYPE, lightType);
        SetUniform<float>((int)RenderKernelArgument_t::SKYBOX_INTENSITY, skyboxIntensity);
        float3 val = float3(eng->m_Camera.position);
        SetUniform<float3>((int)RenderKernelArgument_t::CAMERA_POS, val);
        val = float3(eng->m_Camera.front);
        SetUniform<float3>((int)RenderKernelArgument_t::CAMERA_FRONT, val);
        val = float3(eng->m_Camera.up);
        SetUniform<float3>((int)RenderKernelArgument_t::CAMERA_UP, val);

        if (!eng->ui->isPaused && !eng->ui->framestepOn)
        {
            size_t globalWorksize = (size_t)eng->ui->window_width * eng->ui->window_height;
            if (shardEnd > shardBegin) m_CLContext->ExecuteKernelRange(m_RenderKernel, shardBegin, shardEnd);
            else m_CLContext->ExecuteKernel(m_RenderKernel, globalWorksize);
            if (displayReadback)
            {
                int st = b2rt_read_pixels_rgba8(m_CLContext->GetContext(), pixels8.data(), sizeof(uint32_t) * globalWorksize);
                if (st) throw CLException(std::string("Failed to read display buffer: ") + b2rt_last_error(m_CLContext->GetContext()), st);
            }
            else m_CLContext->ReadBuffer(m_OutputBuffer, pixels.data(), sizeof(float3) * globalWorksize);
            m_CLContext->Finish();
        }
        eng->ui->firstRun = false;
        ++m_FrameCount;
    }

    void CLRaytracer::TraceClosest(const b2rt_ray* rays, uint64_t n, b2rt_hit* hits)
    {
        int st = b2rt_trace_closest(m_CLContext->GetContext(), rays, n, hits);
        if (st) throw CLException(std::string("Failed to trace rays: ") + b2rt_last_error(m_CLContext->GetContext()), st);
    }
    void CLRaytracer::TraceAny(const b2rt_ray* rays, uint64_t n, uint32_t* occluded)
    {
        int st = b2rt_trace_any(m_CLContext->GetContext(), rays, n, occluded);
        if (st) throw CLException(std::string("Failed to trace rays: ") + b2rt_last_error(m_CLContext->GetContext()), st);
    }
    void CLRaytracer::TraceMulti(const b2rt_ray* rays, uint64_t n, uint32_t k, b2rt_hit* hits)
    {
        int st = b2rt_trace_multi(m_CLContext->GetContext(), rays, n, k, hits);
        if (st) throw CLException(std::string("Failed to trace rays: ") + b2rt_last_error(m_CLContext->GetContext()), st);
    }
    void CLRaytracer::ClosestPoint(const b2rt_point_query* queries, uint64_t n, b2rt_point_hit* out)
    {
        int st = b2rt_closest_point(m_CLContext->GetContext(), queries, n, out);
        if (st) throw CLException(std::string("Failed to query closest points: ") + b2rt_last_error(m_CLContext->GetContext()), st);
    }
    void CLRaytracer::TraceRadiance(const b2rt_ray* rays, const uint32_t* seeds, uint64_t n, b2rt_radiance* out)
    {
        int st = b2rt_trace_radiance(m_CLContext->GetContext(), rays, seeds, n, out);
        if (st) throw CLException(std::string("Failed to trace radiance: ") + b2rt_last_error(m_CLContext->GetContext()), st);
    }

    // ---- CLEngineBase (headless) -------------------------------------------------------------------
    CLEngineBase::CLEngineBase()
    {
        render = std::make_shared<CLRaytracer>();
        ui = std::make_shared<CLui>();
    }
    void CLEngineBase::init() { isInitialized = true; }

    void CLEngineBase::renderLoop(const std::string& scene, unsigned int frames, unsigned int maxPrimitives)
    {
        if (!isInitialized) init();
        render->Init();
        render->m_Scene = std::make_shared<CLBVHScene>();
        if (sceneCache)
        {
            CLOBJloader::LoadCached(*render->m_Scene, scene.c_str(), maxPrimitives);
            render->m_Scene->SetupBuffers();
        }
        else
        {
            CLOBJloader loader;
            loader.Load(scene.c_str(), maxPrimitives);
            render->m_Scene->CreateBVHTrees(maxPrimitives);
        }
        for (unsigned int f = 0; f < frames && !windowClose; ++f)
        {
            auto t0 = std::chrono::steady_clock::now();
            processInput();
            render->RenderFrame();
            std::chrono::duration<float> dt = std::chrono::steady_clock::now() - t0;
            FPS = dt.count() > 0 ? 1.0f / dt.count() : 0.0f;
        }
    }
}
