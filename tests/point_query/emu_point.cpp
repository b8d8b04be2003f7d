// emu_point.cpp -- TEST ONLY. The host emulation of tests/emu/emu.cpp (included as it stands: emu_build, ...) plus the
// product's closest-point walk (csrc/point_query.cuh) on the host, and a direct check of the culling lemma that makes the
// walk exact: every child's lb is at most the smallest d2 of the triangles below it.
#include "../emu/emu.cpp"
#include "point_query.cuh"

struct EmuQuery { float x, y, z, max_d2; };

extern "C" void emu_closest_point(const EmuQuery* q, uint64_t n, PointHit* out, EmuStats* st) {
    const U4* wide = reinterpret_cast<const U4*>(g_bvh.nodes.data());
    const U4* leaf = g_bvh.leaf.data();
    for (uint64_t i = 0; i < n; ++i) {
        PointCounters c = { 0, 0, 0, 0, 0 };
        bool overflow = false;
        out[i] = closest_point_wide<true, 256>(wide, leaf, q[i].x, q[i].y, q[i].z, q[i].max_d2, &c, &overflow);
        if (overflow) st->overflow++;
        if (c.max_stack > st->max_stack) st->max_stack = c.max_stack;
        st->wide_visits += c.wide_nodes; st->leaf_blocks += c.leaf_blocks; st->tri_tests += c.tri_tests; st->words += c.words;
    }
}

// The smallest d2 below wide node `index`; counts the children whose lb exceeds the smallest d2 below them.
static float min_below(const U4* wide, const U4* leaf, uint32_t index, float px, float py, float pz, uint64_t& violations,
                       uint64_t& children) {
    const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * index;
    const U4 w0 = p[0], w1 = p[1], w2 = p[2], w3 = p[3], w4 = p[4];
    float lb[8];
    wide_child_lbs(w0, w2, w3, w4, px, py, pz, lb);
    float m = INFINITY;
    for (uint32_t c = 0; c < (w0.w >> 24); ++c) {
        const uint32_t ref = slot_ref(w1, c);
        float below;
        if (ref & REF_LEAF_BIT) {
            PointHit h = { INFINITY, 0.0f, 0.0f, 0xFFFFFFFFu };
            point_leaf<false>(leaf, ref & ~REF_LEAF_BIT, px, py, pz, h, nullptr);
            below = h.d2;
        } else {
            below = min_below(wide, leaf, ref, px, py, pz, violations, children);
        }
        ++children;
        if (!(lb[c] <= below)) ++violations;
        if (below < m) m = below;
    }
    return m;
}

// Over every query (NaN coordinates skipped): children checked and children whose lb exceeds the smallest d2 below (must be 0).
extern "C" void emu_point_lb_check(const EmuQuery* q, uint64_t n, uint64_t* violations, uint64_t* children) {
    const U4* wide = reinterpret_cast<const U4*>(g_bvh.nodes.data());
    const U4* leaf = g_bvh.leaf.data();
    uint64_t v = 0, c = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (!(q[i].x == q[i].x && q[i].y == q[i].y && q[i].z == q[i].z)) continue;
        min_below(wide, leaf, 0, q[i].x, q[i].y, q[i].z, v, c);
    }
    *violations = v;
    *children = c;
}

// The distance routine alone, for the CPU tests of the contract: out = (d2, u, v) per triangle (a, b, c) and point p.
extern "C" void emu_closest_on_triangle(const float* p, const float* abc, uint64_t n, float* out) {
    for (uint64_t i = 0; i < n; ++i) {
        const float* t = abc + 9 * i;
        const float* x = p + 3 * i;
        closest_on_triangle(x[0], x[1], x[2], t[0], t[1], t[2], t[3], t[4], t[5], t[6], t[7], t[8], out[3 * i], out[3 * i + 1], out[3 * i + 2]);
    }
}
