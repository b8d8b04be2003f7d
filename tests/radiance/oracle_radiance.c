/* oracle_radiance.c -- TEST INFRASTRUCTURE ONLY: the contract of b2rt_trace_radiance (include/b2rt.h) on the CPU. It is
 * the oracle's own path loop (oracle/rt_oracle.c render_path, kernel_bvh.cl:349-384) with two differences the contract
 * names: segment 0 is intersected with the ray's tmax instead of 100000, and an out-of-range mtlIndex takes the last
 * material, as the frame kernels do. powf / sinf / cosf are the kernels' (tests/frame_oracle/oracle_devlibm.c, which
 * includes the oracle unchanged), so the GPU records must equal these bit for bit. Compile like the oracle:
 *   gcc -std=c99 -O2 -ffp-contract=off -fno-fast-math -pthread                                                           */
#include "../frame_oracle/oracle_devlibm.c"

typedef struct { float r, g, b; uint32_t seed; } OrRadiance;

static V3 radiance_path(Ray* ray, float tmax, const OrTriangle* tris, const OrNode* nodes, const OrMaterial* mats, uint32_t n_mats,
                        int32_t bounces, int light_type, float sky, uint32_t* seed) {
    V3 radiance = v3(0, 0, 0), beta = v3(1, 1, 1);
    for (int32_t i = 0; i < bounces; ++i) {
        Isect is = intersect(ray, tris, nodes, tmax, 0, NULL);
        tmax = 100000.0f;                                             /* later segments: kernel_bvh.cl:355 */
        if (!is.hit) {
            radiance = add(radiance, mul(beta, scale(v3(0.5f, 0.5f, 0.5f), sky)));
            break;
        }
        uint32_t mi = is.object->mtlIndex;
        if (mi >= n_mats) mi = n_mats - 1u;
        const OrMaterial* m = &mats[mi];
        radiance = add(radiance, scale(mul(beta, ld(&m->emission)), 50.0f));
        V3 wi = v3(0, 0, 0), wo = neg(ray->dir);
        float pdf = 0.0f;
        V3 f = sample_brdf(wo, &wi, &pdf, is.normal, m, seed);
        if (pdf <= 0.0f || pdf != pdf) break;
        beta = mul(beta, sdiv(scale(f, dot(wi, is.normal)), pdf));
        float lp = light_pixel(ray, light_type, &is);
        radiance = add(radiance, mul(mul(v3(lp, lp, lp), ld(&m->diffuse)), beta));
        *ray = init_ray(add(is.pos, scale(wi, 0.01f)), wi);
    }
    return v3(fmax_cl(radiance.x, 0.0f), fmax_cl(radiance.y, 0.0f), fmax_cl(radiance.z, 0.0f));
}

typedef struct {
    const OrTriangle* tris; const OrNode* nodes; const OrMaterial* mats; uint32_t n_mats;
    const OrRay* rays; const uint32_t* seeds; OrRadiance* out;
    int32_t bounces, light_type; float sky; int reference_loop;
} RadCtx;

static void radiance_range(uint64_t lo, uint64_t hi, void* p, int worker) {
    (void)worker;
    const RadCtx* c = (const RadCtx*)p;
    for (uint64_t i = lo; i < hi; ++i) {
        const OrRay* q = &c->rays[i];
        Ray r = init_ray(v3(q->ox, q->oy, q->oz), v3(q->dx, q->dy, q->dz));
        uint32_t seed = c->seeds[i];
        V3 rad = c->reference_loop ? render_path(&r, c->tris, c->nodes, c->mats, (uint32_t)c->bounces, c->light_type, c->sky, &seed)
                                   : radiance_path(&r, q->tmax, c->tris, c->nodes, c->mats, c->n_mats, c->bounces, c->light_type, c->sky, &seed);
        OrRadiance o = { rad.x, rad.y, rad.z, seed };
        c->out[i] = o;
    }
}

static void run(const OrTriangle* tris, const OrNode* nodes, const OrMaterial* mats, uint32_t n_mats, const OrRay* rays,
                const uint32_t* seeds, uint64_t n, int32_t bounces, int32_t light_type, float sky, OrRadiance* out, int threads,
                int reference_loop) {
    RadCtx c = { tris, nodes, mats, n_mats, rays, seeds, out, bounces, light_type, sky, reference_loop };
    parallel_ranges(0, n, threads, radiance_range, &c);
}

/* The contract: out[i] = {radiance, RNG state after the path} of the path started from rays[i] with seeds[i]. */
void oracle_radiance(const OrTriangle* tris, const OrNode* nodes, const OrMaterial* mats, uint32_t n_mats, const OrRay* rays,
                     const uint32_t* seeds, uint64_t n, int32_t bounces, int32_t light_type, float sky, OrRadiance* out, int threads) {
    run(tris, nodes, mats, n_mats, rays, seeds, n, bounces, light_type, sky, out, threads, 0);
}

/* The oracle's own render_path from the same rays (its 100000 on every segment, mtlIndex unclamped), for comparison. */
void oracle_render_path(const OrTriangle* tris, const OrNode* nodes, const OrMaterial* mats, const OrRay* rays, const uint32_t* seeds,
                        uint64_t n, int32_t bounces, int32_t light_type, float sky, OrRadiance* out, int threads) {
    run(tris, nodes, mats, 0, rays, seeds, n, bounces, light_type, sky, out, threads, 1);
}
