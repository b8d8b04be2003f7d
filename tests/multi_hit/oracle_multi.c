/* oracle_multi.c -- TEST INFRASTRUCTURE ONLY: the k nearest hits per ray (the contract of b2rt_trace_multi, include/b2rt.h)
 * on the CPU. It is the oracle's reference walk, Intersect() of kernel_bvh.cl:171-219, with isect replaced by a sorted list
 * of at most k hits. oracle/rt_oracle.c is included as it stands, so InitRay, RayBounds and RayTriangle are the very
 * functions behind oracle_trace_closest; nothing is taken from the product. Compile like the oracle:
 *   gcc -std=c99 -O2 -ffp-contract=off -fno-fast-math -pthread                                                      */
#include "../../oracle/rt_oracle.c"

/* row[0, k) receives the list, padded with {tmax, 0, 0, miss}. */
static void intersect_multi(const Ray* ray, const OrTriangle* tris, const OrNode* nodes, float tmax, uint32_t k, OrHit* row) {
    uint32_t count = 0;
    float bound = tmax;                       /* tmax until the list is full, then the t of its k-th entry */
    int cap = 64, top = 0, cur = 0;
    int local[64];
    int* stack = local;
    for (;;) {
        const OrNode* node = &nodes[cur];
        if (ray_bounds(node, ray, bound)) {
            if (node->nPrimitives > 0) {
                for (int i = 0; i < node->nPrimitives; ++i) {
                    Isect is;
                    memset(&is, 0, sizeof(is));
                    is.t = bound;
                    ray_triangle(ray, &tris[node->offset + i], &is);          /* accepts iff t < bound */
                    if (!is.hit) continue;
                    /* after every entry with t <= is.t; a full list drops its last entry */
                    uint32_t j = count < k ? count : k - 1;
                    while (j > 0 && row[j - 1].t > is.t) { row[j] = row[j - 1]; --j; }
                    row[j].t = is.t; row[j].u = is.u; row[j].v = is.v; row[j].tri = node->offset + (uint32_t)i;
                    if (count < k) ++count;
                    if (count == k) bound = row[k - 1].t;
                }
                if (top == 0) break;
                cur = stack[--top];
            } else {
                if (top == cap) {
                    int* bigger = (int*)malloc(sizeof(int) * cap * 2);
                    memcpy(bigger, stack, sizeof(int) * cap);
                    if (stack != local) free(stack);
                    stack = bigger;
                    cap *= 2;
                }
                if (ray->sign[node->axis]) {                       /* :200-203 */
                    stack[top++] = cur + 1;
                    cur = (int)node->offset;
                } else {                                           /* :204-207 */
                    stack[top++] = (int)node->offset;
                    cur = cur + 1;
                }
            }
        } else {
            if (top == 0) break;
            cur = stack[--top];
        }
    }
    if (stack != local) free(stack);
    for (uint32_t i = count; i < k; ++i) { row[i].t = tmax; row[i].u = 0.0f; row[i].v = 0.0f; row[i].tri = 0xFFFFFFFFu; }
}

typedef struct { const OrTriangle* tris; const OrNode* nodes; const OrRay* rays; uint32_t k; OrHit* hits; } MultiCtx;

static void multi_range(uint64_t lo, uint64_t hi, void* p, int worker) {
    (void)worker;
    MultiCtx* c = (MultiCtx*)p;
    for (uint64_t i = lo; i < hi; ++i) {
        const OrRay* q = &c->rays[i];
        Ray r = init_ray(v3(q->ox, q->oy, q->oz), v3(q->dx, q->dy, q->dz));
        intersect_multi(&r, c->tris, c->nodes, q->tmax, c->k, c->hits + i * c->k);
    }
}

/* hits: OrHit[n * k], row i = the k nearest hits of ray i. k >= 1. threads <= 0 -> all hardware threads. */
void oracle_trace_multi(const OrTriangle* tris, const OrNode* nodes, const OrRay* rays, uint64_t n, uint32_t k, OrHit* hits,
                        int threads) {
    MultiCtx c = { tris, nodes, rays, k, hits };
    parallel_ranges(0, n, threads, multi_range, &c);
}
