/* oracle_point.c -- TEST INFRASTRUCTURE ONLY: the contract of b2rt_closest_point (include/b2rt.h) restated by brute force
 * over the scene's CLTriangle array: every triangle is a candidate, the smallest (d2, tri) with d2 <= max_d2 wins.
 * Nothing is taken from the product's sources. Compile with
 *   gcc -std=c99 -O2 -ffp-contract=off -fno-fast-math -pthread
 * so that every float operation below is one IEEE fp32 operation rounded to nearest. */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

typedef struct { float x, y, z, max_d2; } Query;
typedef struct { float d2, u, v; uint32_t tri; } PHit;

static float dot3(float ax, float ay, float az, float bx, float by, float bz) { return (ax * bx + ay * by) + az * bz; }
static float clamp01(float t) { return t > 0.0f ? (t < 1.0f ? t : 1.0f) : 0.0f; }
/* per axis into [lo, hi]; NaN becomes lo */
static float clampq(float q, float lo, float hi) { return fminf(fmaxf(q, lo), hi); }
static float dist2(const float p[3], const float q[3]) {
    const float dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
    return (dx * dx + dy * dy) + dz * dz;
}

/* Ericson, Real-Time Collision Detection 5.1.5, with the contract's degenerate fallback and vertex-box clamp. */
void oracle_closest_on_triangle(const float p[3], const float a[3], const float b[3], const float c[3], float out[3]) {
    float ab[3], ac[3], ap[3], bp[3], cp[3], cb[3], lo[3], hi[3], q[3];
    for (int i = 0; i < 3; ++i) {
        ab[i] = b[i] - a[i]; ac[i] = c[i] - a[i]; ap[i] = p[i] - a[i];
        bp[i] = p[i] - b[i]; cp[i] = p[i] - c[i]; cb[i] = c[i] - b[i];
        lo[i] = fminf(fminf(a[i], b[i]), c[i]); hi[i] = fmaxf(fmaxf(a[i], b[i]), c[i]);
    }
    const float d1 = dot3(ab[0], ab[1], ab[2], ap[0], ap[1], ap[2]);
    const float d2 = dot3(ac[0], ac[1], ac[2], ap[0], ap[1], ap[2]);
    const float d3 = dot3(ab[0], ab[1], ab[2], bp[0], bp[1], bp[2]);
    const float d4 = dot3(ac[0], ac[1], ac[2], bp[0], bp[1], bp[2]);
    const float d5 = dot3(ab[0], ab[1], ab[2], cp[0], cp[1], cp[2]);
    const float d6 = dot3(ac[0], ac[1], ac[2], cp[0], cp[1], cp[2]);
    const float vc = d1 * d4 - d3 * d2, vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
    float u, v;
    if (d1 <= 0.0f && d2 <= 0.0f) { for (int i = 0; i < 3; ++i) q[i] = a[i]; u = 0.0f; v = 0.0f; }
    else if (d3 >= 0.0f && d4 <= d3) { for (int i = 0; i < 3; ++i) q[i] = b[i]; u = 1.0f; v = 0.0f; }
    else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f && d1 - d3 > 0.0f) {
        const float t = d1 / (d1 - d3);
        for (int i = 0; i < 3; ++i) q[i] = a[i] + ab[i] * t;
        u = t; v = 0.0f;
    } else if (d6 >= 0.0f && d5 <= d6) { for (int i = 0; i < 3; ++i) q[i] = c[i]; u = 0.0f; v = 1.0f; }
    else if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f && d2 - d6 > 0.0f) {
        const float t = d2 / (d2 - d6);
        for (int i = 0; i < 3; ++i) q[i] = a[i] + ac[i] * t;
        u = 0.0f; v = t;
    } else if (va <= 0.0f && (d4 - d3) >= 0.0f && (d5 - d6) >= 0.0f && (d4 - d3) + (d5 - d6) > 0.0f) {
        const float t = (d4 - d3) / ((d4 - d3) + (d5 - d6));
        for (int i = 0; i < 3; ++i) q[i] = b[i] + cb[i] * t;
        u = 1.0f - t; v = t;
    } else if ((va + vb) + vc > 0.0f) {
        const float denom = 1.0f / ((va + vb) + vc);
        const float w1 = vb * denom, w2 = vc * denom;
        for (int i = 0; i < 3; ++i) q[i] = (a[i] + ab[i] * w1) + ac[i] * w2;
        u = w1; v = w2;
    } else {
        /* degenerate: edges ab, ac, bc from their origins a, a, b; smallest clamped d2, ties to the earlier edge */
        const float* org[3] = { a, a, b };
        const float* e[3] = { ab, ac, cb };
        const float* op[3] = { ap, ap, bp };
        float best = 0.0f, bu = 0.0f, bv = 0.0f;
        for (int k = 0; k < 3; ++k) {
            const float t = clamp01(dot3(op[k][0], op[k][1], op[k][2], e[k][0], e[k][1], e[k][2]) /
                                    dot3(e[k][0], e[k][1], e[k][2], e[k][0], e[k][1], e[k][2]));
            float qq[3];
            for (int i = 0; i < 3; ++i) qq[i] = clampq(org[k][i] + e[k][i] * t, lo[i], hi[i]);
            const float dd = dist2(p, qq);
            if (k == 0 || dd < best) {
                best = dd;
                bu = k == 0 ? t : (k == 1 ? 0.0f : 1.0f - t);
                bv = k == 0 ? 0.0f : t;
            }
        }
        out[0] = best; out[1] = bu; out[2] = bv;
        return;
    }
    for (int i = 0; i < 3; ++i) q[i] = clampq(q[i], lo[i], hi[i]);
    out[0] = dist2(p, q); out[1] = u; out[2] = v;
}

static void position(const uint8_t* tri, int vertex, float out[3]) { memcpy(out, tri + 80 * vertex, 12); }

static PHit query_one(const uint8_t* tris, uint64_t n_tris, const Query* q) {
    PHit h = { q->max_d2, 0.0f, 0.0f, 0xFFFFFFFFu };
    if (isnan(q->x) || isnan(q->y) || isnan(q->z) || !(q->max_d2 >= 0.0f)) return h;
    const float p[3] = { q->x, q->y, q->z };
    for (uint64_t k = 0; k < n_tris; ++k) {
        float a[3], b[3], c[3], r[3];
        position(tris + 256 * k, 0, a); position(tris + 256 * k, 1, b); position(tris + 256 * k, 2, c);
        oracle_closest_on_triangle(p, a, b, c, r);
        /* strict <: with ties the smaller index, which is visited first, stays */
        if (r[0] <= q->max_d2 && (h.tri == 0xFFFFFFFFu || r[0] < h.d2)) { h.d2 = r[0]; h.u = r[1]; h.v = r[2]; h.tri = (uint32_t)k; }
    }
    return h;
}

typedef struct { const uint8_t* tris; uint64_t n_tris; const Query* q; PHit* out; uint64_t lo, hi; } Part;

static void* run_part(void* arg) {
    Part* p = (Part*)arg;
    for (uint64_t i = p->lo; i < p->hi; ++i) p->out[i] = query_one(p->tris, p->n_tris, &p->q[i]);
    return NULL;
}

/* out[i] = the contract's record for q[i]; threads <= 0: one per online CPU (at most 64). */
void oracle_closest_point(const void* tris, uint64_t n_tris, const void* queries, uint64_t n, void* out, int threads) {
    if (threads <= 0) threads = (int)sysconf(_SC_NPROCESSORS_ONLN);
    if (threads < 1) threads = 1;
    if (threads > 64) threads = 64;
    if ((uint64_t)threads > n) threads = n ? (int)n : 1;
    pthread_t th[64];
    Part parts[64];
    for (int w = 0; w < threads; ++w) {
        parts[w] = (Part){ (const uint8_t*)tris, n_tris, (const Query*)queries, (PHit*)out, n * (uint64_t)w / (uint64_t)threads,
                           n * (uint64_t)(w + 1) / (uint64_t)threads };
        pthread_create(&th[w], NULL, run_part, &parts[w]);
    }
    for (int w = 0; w < threads; ++w) pthread_join(th[w], NULL);
}
