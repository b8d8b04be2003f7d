// point_query.cuh -- closest point on the scene's triangles (b2rt_closest_point, include/b2rt.h) over the compressed wide
// BVH. Like traverse.cuh, the same text compiles for the sm_100a kernels (kernels.cu) and, TEST ONLY, as plain C++ for the
// host emulation (tests/point_query/emu_point.cpp).
//
// Exactness (DESIGN.md 4e): every fp32 operation of the distance and of the lower bounds is one explicit IEEE operation
// rounded to nearest (xadd / xsub / xmul / xdiv: __f*_rn on the device, which nvcc never contracts), except the plane
// decode, which rounds outwards on purpose (fma_rd / fma_ru). No packed pairs are used: a packed product feeding a packed
// sum would be contracted into FFMA2 (traverse.cuh, "packed fp32 pairs"), and a contracted lb or d2 breaks lb <= d2.
// tests/test_point_query_oracle.py checks the SASS.
//   lb(child) = (gx*gx + gy*gy) + gz*gz,   g = max(lo - p, p - hi, 0) on the child's quantised box decoded outwards
//   d2(tri)   = (dx*dx + dy*dy) + dz*dz,   d = p - q,  q = the region test's point clamped into the triangle's vertex box
// Quantised box >= binary node box >= leaf box >= every vertex box below, and fp32 subtraction, squaring and addition are
// monotone, so lb(child) <= d2 of every triangle below it. A child is skipped iff !(lb <= best): the minimum of the total
// order (d2, tri) is never skipped, whatever the visiting order.
#pragma once
#include "traverse.cuh"

namespace b2rt {

struct PointHit { float d2, u, v; uint32_t tri; };        // b2rt_point_hit
struct PointCounters { uint32_t wide_nodes, leaf_blocks, tri_tests, words, max_stack; };

B2_HD float dot3_rn(float ax, float ay, float az, float bx, float by, float bz) {
    return xadd(xadd(xmul(ax, bx), xmul(ay, by)), xmul(az, bz));
}
B2_HD float clamp01(float t) { return t > 0.0f ? (t < 1.0f ? t : 1.0f) : 0.0f; }   // NaN -> 0
// q clamped into [lo, hi]; a NaN q becomes lo (max_nn ignores NaN)
B2_HD float clamp_box(float q, float lo, float hi) { return min_nn(max_nn(q, lo), hi); }
B2_HD float dist2(float px, float py, float pz, float qx, float qy, float qz) {
    const float dx = xsub(px, qx), dy = xsub(py, qy), dz = xsub(pz, qz);
    return xadd(xadd(xmul(dx, dx), xmul(dy, dy)), xmul(dz, dz));
}

// The closest point of triangle (a, b, c) to p: Ericson, "Real-Time Collision Detection" 5.1.5, in the contract's operation
// order (b2rt.h). An edge region also requires its denominator to be > 0: a zero-length edge (repeated vertex) would
// otherwise take the edge branch with t = 0/0. d2 of the point clamped into the vertex box; (u, v) in the reference's barycentric convention,
// point = (1-u-v) a + u b + v c.
B2_HD void closest_on_triangle(float px, float py, float pz, float ax, float ay, float az, float bx, float by, float bz,
                               float cx, float cy, float cz, float& d2, float& u, float& v) {
    const float abx = xsub(bx, ax), aby = xsub(by, ay), abz = xsub(bz, az);
    const float acx = xsub(cx, ax), acy = xsub(cy, ay), acz = xsub(cz, az);
    const float apx = xsub(px, ax), apy = xsub(py, ay), apz = xsub(pz, az);
    const float d1 = dot3_rn(abx, aby, abz, apx, apy, apz), e2 = dot3_rn(acx, acy, acz, apx, apy, apz);
    const float bpx = xsub(px, bx), bpy = xsub(py, by), bpz = xsub(pz, bz);
    const float cpx = xsub(px, cx), cpy = xsub(py, cy), cpz = xsub(pz, cz);
    const float d3 = dot3_rn(abx, aby, abz, bpx, bpy, bpz), d4 = dot3_rn(acx, acy, acz, bpx, bpy, bpz);
    const float d5 = dot3_rn(abx, aby, abz, cpx, cpy, cpz), d6 = dot3_rn(acx, acy, acz, cpx, cpy, cpz);
    const float vc = xsub(xmul(d1, d4), xmul(d3, e2));
    const float vb = xsub(xmul(d5, e2), xmul(d1, d6));
    const float va = xsub(xmul(d3, d6), xmul(d5, d4));
    const float lox = min_nn(min_nn(ax, bx), cx), loy = min_nn(min_nn(ay, by), cy), loz = min_nn(min_nn(az, bz), cz);
    const float hix = max_nn(max_nn(ax, bx), cx), hiy = max_nn(max_nn(ay, by), cy), hiz = max_nn(max_nn(az, bz), cz);
    float qx, qy, qz;
    if (d1 <= 0.0f && e2 <= 0.0f) { qx = ax; qy = ay; qz = az; u = 0.0f; v = 0.0f; }                          // vertex a
    else if (d3 >= 0.0f && d4 <= d3) { qx = bx; qy = by; qz = bz; u = 1.0f; v = 0.0f; }                      // vertex b
    else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f && xsub(d1, d3) > 0.0f) {                               // edge ab
        const float t = xdiv(d1, xsub(d1, d3));
        qx = xadd(ax, xmul(abx, t)); qy = xadd(ay, xmul(aby, t)); qz = xadd(az, xmul(abz, t)); u = t; v = 0.0f;
    } else if (d6 >= 0.0f && d5 <= d6) { qx = cx; qy = cy; qz = cz; u = 0.0f; v = 1.0f; }                    // vertex c
    else if (vb <= 0.0f && e2 >= 0.0f && d6 <= 0.0f && xsub(e2, d6) > 0.0f) {                               // edge ac
        const float t = xdiv(e2, xsub(e2, d6));
        qx = xadd(ax, xmul(acx, t)); qy = xadd(ay, xmul(acy, t)); qz = xadd(az, xmul(acz, t)); u = 0.0f; v = t;
    } else if (va <= 0.0f && xsub(d4, d3) >= 0.0f && xsub(d5, d6) >= 0.0f && xadd(xsub(d4, d3), xsub(d5, d6)) > 0.0f) {   // edge bc
        const float n43 = xsub(d4, d3);
        const float t = xdiv(n43, xadd(n43, xsub(d5, d6)));
        qx = xadd(bx, xmul(xsub(cx, bx), t)); qy = xadd(by, xmul(xsub(cy, by), t)); qz = xadd(bz, xmul(xsub(cz, bz), t));
        u = xsub(1.0f, t); v = t;
    } else {
        const float sum = xadd(xadd(va, vb), vc);
        if (sum > 0.0f) {                                                                                      // interior
            const float denom = xdiv(1.0f, sum);
            const float wv = xmul(vb, denom), ww = xmul(vc, denom);
            qx = xadd(xadd(ax, xmul(abx, wv)), xmul(acx, ww));
            qy = xadd(xadd(ay, xmul(aby, wv)), xmul(acy, ww));
            qz = xadd(xadd(az, xmul(abz, wv)), xmul(acz, ww));
            u = wv; v = ww;
        } else {
            // degenerate (zero-area, collinear or non-finite region values): the three edges ab, ac, bc in this order,
            // t = clamp01(op.e / e.e) from the edge's origin o; the smallest clamped d2 wins, ties to the earlier edge
            const float cbx = xsub(cx, bx), cby = xsub(cy, by), cbz = xsub(cz, bz);
            const float t0 = clamp01(xdiv(d1, dot3_rn(abx, aby, abz, abx, aby, abz)));
            const float t1 = clamp01(xdiv(e2, dot3_rn(acx, acy, acz, acx, acy, acz)));
            const float t2 = clamp01(xdiv(dot3_rn(bpx, bpy, bpz, cbx, cby, cbz), dot3_rn(cbx, cby, cbz, cbx, cby, cbz)));
            const float e0 = dist2(px, py, pz, clamp_box(xadd(ax, xmul(abx, t0)), lox, hix), clamp_box(xadd(ay, xmul(aby, t0)), loy, hiy),
                                   clamp_box(xadd(az, xmul(abz, t0)), loz, hiz));
            const float e1 = dist2(px, py, pz, clamp_box(xadd(ax, xmul(acx, t1)), lox, hix), clamp_box(xadd(ay, xmul(acy, t1)), loy, hiy),
                                   clamp_box(xadd(az, xmul(acz, t1)), loz, hiz));
            const float e3 = dist2(px, py, pz, clamp_box(xadd(bx, xmul(cbx, t2)), lox, hix), clamp_box(xadd(by, xmul(cby, t2)), loy, hiy),
                                   clamp_box(xadd(bz, xmul(cbz, t2)), loz, hiz));
            d2 = e0; u = t0; v = 0.0f;
            if (e1 < d2) { d2 = e1; u = 0.0f; v = t1; }
            if (e3 < d2) { d2 = e3; u = xsub(1.0f, t2); v = t2; }
            return;
        }
    }
    d2 = dist2(px, py, pz, clamp_box(qx, lox, hix), clamp_box(qy, loy, hiy), clamp_box(qz, loz, hiz));
}

// Candidate (d2, tri) replaces the best so far iff it is smaller in the total order (d2, tri). best starts as
// {max_d2, 0, 0, MISS}, so a candidate is only ever taken with d2 <= max_d2.
B2_HD void point_take(PointHit& best, float d2, float u, float v, uint32_t tri) {
    if (d2 < best.d2 || (d2 == best.d2 && tri < best.tri)) { best.d2 = d2; best.u = u; best.v = v; best.tri = tri; }
}

// Lower bound of d2 for a box [lo, hi]: per axis the gap g = max(lo - p, p - hi, 0), then d2's squares and summation order.
B2_HD float box_lb(float px, float py, float pz, float lox, float loy, float loz, float hix, float hiy, float hiz) {
    const float gx = max_nn(max_nn(xsub(lox, px), xsub(px, hix)), 0.0f);
    const float gy = max_nn(max_nn(xsub(loy, py), xsub(py, hiy)), 0.0f);
    const float gz = max_nn(max_nn(xsub(loz, pz), xsub(pz, hiz)), 0.0f);
    return xadd(xadd(xmul(gx, gx), xmul(gy, gy)), xmul(gz, gz));
}

// lb of every child slot of a loaded wide node (slots >= n_children: +inf, which still passes best = +inf: mask them). The planes are decoded outwards like
// test_wide_node_robust: lo = fma_rd(q, S, base) <= the child's exact lo, hi = fma_ru(q, S, base) >= its exact hi.
B2_HD void wide_child_lbs(const U4& w0, const U4& w2, const U4& w3, const U4& w4, float px, float py, float pz, float lb[8]) {
    const uint32_t qlo_a[3] = { w2.x, w2.z, w3.x }, qlo_b[3] = { w2.y, w2.w, w3.y };   // slots 0..3 / 4..7
    const uint32_t qhi_a[3] = { w3.z, w4.x, w4.z }, qhi_b[3] = { w3.w, w4.y, w4.w };
    const float base[3] = { bits2f(w0.x), bits2f(w0.y), bits2f(w0.z) };
    const float S[3] = { bits2f((w0.w & 0xffu) << 23), bits2f(((w0.w >> 8) & 0xffu) << 23), bits2f(((w0.w >> 16) & 0xffu) << 23) };
    const uint32_t n_children = w0.w >> 24;
#pragma unroll
    for (uint32_t c = 0; c < 8; ++c) {
        float lo[3], hi[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const uint32_t ql = c < 4 ? byte_of(qlo_a[a], c) : byte_of(qlo_b[a], c - 4);
            const uint32_t qh = c < 4 ? byte_of(qhi_a[a], c) : byte_of(qhi_b[a], c - 4);
            lo[a] = fma_rd(u2f(ql), S[a], base[a]);
            hi[a] = fma_ru(u2f(qh), S[a], base[a]);
        }
        const float l = box_lb(px, py, pz, lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]);
        lb[c] = c < n_children ? l : INFINITY;
    }
}

// Child reference of slot c: wide node index, or REF_LEAF_BIT | leaf block offset (see b2rt_types.h).
B2_HD uint32_t slot_ref(const U4& w1, uint32_t c) {
    const uint32_t m = byte_of(c < 4 ? w1.z : w1.w, c & 3u);
    return (m & META_INTERIOR) ? w1.x + (m & META_MAX_LEAF_OFFSET) : (REF_LEAF_BIT | (w1.y + m));
}

// Every triangle of one leaf block against p; the loader's second copy of a face (flags) is its own candidate id + 1,
// evaluated with its vertices rotated as stored, like visit_leaf does for rays.
template <bool COUNT>
B2_HD void point_leaf(const U4* leaf, uint32_t offset, float px, float py, float pz, PointHit& best, PointCounters* c) {
    const U4* p = leaf + offset;
    U4 a = ld128(p), b = ld128(p + 1), cc = ld128(p + 2);
    const uint32_t nrec = (a.w >> LEAF_NREC_SHIFT) & LEAF_NREC_MASK;
    if (COUNT) { c->leaf_blocks++; c->words += LEAF_RECORD_WORDS * nrec; }
    uint32_t id = b.w;
    for (uint32_t k = 0;;) {
        const float v1x = bits2f(a.x), v1y = bits2f(a.y), v1z = bits2f(a.z);
        const float v2x = bits2f(b.x), v2y = bits2f(b.y), v2z = bits2f(b.z);
        const float v3x = bits2f(cc.x), v3y = bits2f(cc.y), v3z = bits2f(cc.z);
        const uint32_t flags = a.w & REC_FLAG_MASK;
        float d2, u, v;
        closest_on_triangle(px, py, pz, v1x, v1y, v1z, v2x, v2y, v2z, v3x, v3y, v3z, d2, u, v);
        point_take(best, d2, u, v, id);
        if (COUNT) c->tri_tests++;
        if (flags) {
            const bool left = flags == REC_ROT_LEFT;       // (v2, v3, v1) or (v3, v1, v2)
            closest_on_triangle(px, py, pz, left ? v2x : v3x, left ? v2y : v3y, left ? v2z : v3z,
                                left ? v3x : v1x, left ? v3y : v1y, left ? v3z : v1z,
                                left ? v1x : v2x, left ? v1y : v2y, left ? v1z : v2z, d2, u, v);
            point_take(best, d2, u, v, id + 1u);
            if (COUNT) c->tri_tests++;
        }
        id += flags ? 2u : 1u;
        if (++k >= nrec) break;
        const U4* q = p + LEAF_RECORD_WORDS * k;
        a = ld128(q); b = ld128(q + 1); cc = ld128(q + 2);
    }
}

// A deferred child: its reference and its lb, so that a pop whose lb exceeds the best so far costs no fetch.
struct PointEntry { uint32_t ref; float lb; };

// One query's walk. `cur` is the next wide node or leaf block to visit (REF_EMPTY: finished). A node step visits the
// surviving children nearest first: the nearest becomes `cur`, the others are pushed farthest first -- all surviving
// children but one, the push discipline of Lane::node_step, so the tree's stack bound (wide_stack_bound) bounds `sp`.
template <bool COUNT, int CAP>
struct PointLane {
    float px, py, pz;
    PointHit best;
    uint32_t cur;
    int sp;
    bool overflow;
    PointCounters tc;

    // false: the query misses without a walk (NaN coordinate, negative or NaN max_d2)
    B2_HD bool start(float x, float y, float z, float max_d2) {
        px = x; py = y; pz = z;
        best.d2 = max_d2; best.u = 0.0f; best.v = 0.0f; best.tri = 0xFFFFFFFFu;
        sp = 0; overflow = false;
        const bool go = x == x && y == y && z == z && max_d2 >= 0.0f;
        cur = go ? 0u : REF_EMPTY;
        return go;
    }
    B2_HD bool done() const { return cur == REF_EMPTY; }
    B2_HD bool wants_node() const { return cur != REF_EMPTY && !(cur & REF_LEAF_BIT); }
    B2_HD bool wants_leaf() const { return cur != REF_EMPTY && (cur & REF_LEAF_BIT); }
    // next deferred entry that can still hold the answer; entries whose lb exceeds best are dropped unread
    B2_HD void pop(const PointEntry* stack) {
        cur = REF_EMPTY;
        while (sp > 0) {
            const PointEntry e = stack[--sp];
            if (e.lb <= best.d2) { cur = e.ref; break; }
        }
    }
    B2_HD void push(PointEntry* stack, uint32_t ref, float lb) {
        if (COUNT && sp >= CAP) { overflow = true; return; }
        stack[sp].ref = ref; stack[sp].lb = lb;
        ++sp;
        if (COUNT && (uint32_t)sp > tc.max_stack) tc.max_stack = (uint32_t)sp;
    }
    B2_HD void node_step(const U4* wide, PointEntry* stack) {
        const U4* p = wide + (uint32_t)WIDE_NODE_WORDS * cur;
        const U4 w0 = ld128(p), w1 = ld128(p + 1), w2 = ld128(p + 2), w3 = ld128(p + 3), w4 = ld128(p + 4);
        if (COUNT) { tc.wide_nodes++; tc.words += WIDE_NODE_WORDS; }
        float lb[8];
        wide_child_lbs(w0, w2, w3, w4, px, py, pz, lb);
        uint32_t mask = 0;
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) mask |= (lb[c] <= best.d2 ? 1u : 0u) << c;
        mask &= low_mask(w0.w >> 24);                      // empty slots (lb = +inf) would pass a bound of +inf
        if (mask == 0) { pop(stack); return; }
        while (mask & (mask - 1u)) {                       // more than one survivor: push the farthest
            uint32_t far = 0;
            float m = -1.0f;
#pragma unroll
            for (uint32_t c = 0; c < 8; ++c)
                if (((mask >> c) & 1u) && !(lb[c] < m)) { m = lb[c]; far = c; }
            push(stack, slot_ref(w1, far), m);
            mask &= ~(1u << far);
        }
        cur = slot_ref(w1, ctz32(mask));
    }
    B2_HD void leaf_step(const U4* leaf, PointEntry* stack) {
        point_leaf<COUNT>(leaf, cur & ~REF_LEAF_BIT, px, py, pz, best, COUNT ? &tc : nullptr);
        pop(stack);
    }
};

// One thread = one query, leaves as soon as they come up (the host emulation; the kernel interleaves by warp vote).
template <bool COUNT, int CAP>
B2_HD PointHit closest_point_wide(const U4* wide, const U4* leaf, float x, float y, float z, float max_d2, PointCounters* c,
                                  bool* overflow) {
    PointLane<COUNT, CAP> L;
    PointEntry stack[CAP];
    L.tc.wide_nodes = L.tc.leaf_blocks = L.tc.tri_tests = L.tc.words = L.tc.max_stack = 0;
    L.start(x, y, z, max_d2);
    while (!L.done()) {
        if (L.wants_leaf()) L.leaf_step(leaf, stack);
        else L.node_step(wide, stack);
    }
    if (COUNT && c) *c = L.tc;
    if (overflow) *overflow = L.overflow;
    return L.best;
}

}  // namespace b2rt
