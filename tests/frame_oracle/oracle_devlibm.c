/* oracle_devlibm.c -- TEST INFRASTRUCTURE ONLY: the oracle (oracle/rt_oracle.c, included as it stands) with powf / sinf /
 * cosf evaluated the way the frame kernels evaluate them (pow_cr / sin_cr / cos_cr, csrc/shade.cuh): in fp64, rounded
 * once to float. Every other operation is the oracle's own fp32 arithmetic, so a GPU frame must equal this one bit for
 * bit; the glibc oracle differs from both by the last ulp of a few powf results. Compile like the oracle:
 *   gcc -std=c99 -O2 -ffp-contract=off -fno-fast-math -pthread
 * fo_run() exposes the oracle's shading functions one record at a time, in the record layout of
 * tests/frame_oracle/shade_probe.cu, which runs the kernels' functions on the same records.                          */
#define _GNU_SOURCE
#include <math.h>
#include <stdint.h>

/* pow_cr of csrc/shade.cuh: the special values of C99 powf that the fp64 route does not produce by itself (x^0 = 1,
 * 1^y = 1), the exact fp64 square for b == 2, else exp2(b log2 a) rounded once */
static float dev_powf(float a, float b) {
    if (b == 0.0f || (a == 1.0f && !(fabsf(b) < INFINITY))) return 1.0f;
    if (b == 2.0f) return (float)((double)a * (double)a);
    return (float)exp2((double)b * log2((double)a));
}
static float dev_sinf(float a) { return (float)sin((double)a); }
static float dev_cosf(float a) { return (float)cos((double)a); }

#define powf dev_powf
#define sinf dev_sinf
#define cosf dev_cosf
#include "../../oracle/rt_oracle.c"          /* the three macros stay: the wrappers below mean the same functions */

/* ---- one record of the shading probe (16 input words -> 16 output words), the layouts of shade_probe.cu ---------- */
enum { FO_POW = 0, FO_SINCOS = 1, FO_FRAME = 2, FO_BRDF = 3, FO_LIGHT = 4, FO_CAMERA = 5, FO_RND = 6, FO_ACCUMULATE = 7 };

typedef union { uint32_t u; float f; int32_t i; } W;

static V3 ldw(const W* w) { return v3(w[0].f, w[1].f, w[2].f); }
static void stw(W* w, V3 v) { w[0].f = v.x; w[1].f = v.y; w[2].f = v.z; }

/* the accumulation of render_range (kernel_bvh.cl:449-455) for one pixel */
static void accumulate_px(float* px, V3 rad, uint32_t frame_count) {
    if (frame_count == 0) {
        px[0] = powf(rad.x, 0.45454545f); px[1] = powf(rad.y, 0.45454545f); px[2] = powf(rad.z, 0.45454545f);
    } else {
        float fm1 = (float)(frame_count - 1), fc = (float)frame_count;
        float in[3] = { px[0], px[1], px[2] }, r[3] = { rad.x, rad.y, rad.z };
        for (int k = 0; k < 3; ++k)
            px[k] = powf((powf(in[k], 2.2f) * fm1 + r[k]) / fc, 0.454545f);
    }
    px[3] = 0.0f;
}

static void fo_record(int op, const W* in, W* out) {
    switch (op) {
    case FO_POW:
        out[0].f = powf(in[0].f, in[1].f);
        break;
    case FO_SINCOS:
        out[0].f = sinf(in[0].f); out[1].f = cosf(in[0].f);
        break;
    case FO_FRAME:
        stw(out, tangent_frame_sample(ldw(in), in[3].f, in[4].f, in[5].f));
        break;
    case FO_BRDF: {
        OrMaterial m;
        memset(&m, 0, sizeof(m));
        m.roughness = in[6].f;
        m.specular.x = in[7].f; m.specular.y = in[8].f; m.specular.z = in[9].f;
        m.diffuse.x = in[10].f; m.diffuse.y = in[11].f; m.diffuse.z = in[12].f;
        uint32_t seed = in[13].u;
        V3 wi = v3(0.0f, 0.0f, 0.0f);
        float pdf = 0.0f;
        stw(out, sample_brdf(ldw(in), &wi, &pdf, ldw(in + 3), &m, &seed));
        stw(out + 3, wi);
        out[6].f = pdf; out[7].u = seed;
        break;
    }
    case FO_LIGHT: {
        Ray r;
        Isect is;
        memset(&r, 0, sizeof(r));
        memset(&is, 0, sizeof(is));
        r.origin = ldw(in); r.dir = ldw(in + 3);
        is.t = in[6].f; is.normal = ldw(in + 7);
        out[0].f = light_pixel(&r, in[10].i, &is);
        break;
    }
    case FO_CAMERA: {
        uint32_t seed = in[3].u;
        Ray r = create_ray(in[2].u, in[0].u, in[1].u, v3(0.0f, 0.0f, 0.0f), ldw(in + 5), ldw(in + 8), &seed);
        stw(out, r.dir);
        out[3].u = seed;
        break;
    }
    case FO_RND: {
        uint32_t seed = in[0].u;
        out[0].f = rnd(&seed); out[1].u = seed;
        out[2].u = hash_u32(in[0].u);
        break;
    }
    case FO_ACCUMULATE: {
        float px[4] = { in[0].f, in[1].f, in[2].f, in[3].f };
        accumulate_px(px, ldw(in + 4), in[7].u);
        for (int k = 0; k < 4; ++k) out[k].f = px[k];
        break;
    }
    default:
        break;
    }
}

/* in, out: n records of 16 words each; out is zeroed before the record is evaluated */
void fo_run(int op, uint64_t n, const uint32_t* in, uint32_t* out) {
    for (uint64_t i = 0; i < n; ++i) {
        W* o = (W*)(out + 16 * i);
        memset(o, 0, 16 * sizeof(uint32_t));
        fo_record(op, (const W*)(in + 16 * i), o);
    }
}

/* the camera's half-angle tangent as create_ray computes it (the product takes it from the host libm as well) */
float fo_camera_angle(void) { return tanf(0.5f * (45.0f * 3.1415f / 180.0f)); }
