// emu_multi.cpp -- TEST ONLY. The host emulation of tests/emu/emu.cpp (included as it stands: emu_build, emu_trace, ...) plus
// the HIT_MULTI policy of the product's Lane (csrc/traverse.cuh) run through trace_wide, so that the k-nearest-hits logic
// of the kernels -- insertion, bound, padding, speculation included -- is checked against the oracle without a GPU.
#include "../emu/emu.cpp"

// hits: EmuHit[n * k]. schedule as for emu_trace: 0 = leaves first, else per-ray pseudo-random node / leaf interleavings.
extern "C" void emu_trace_multi(const EmuRay* rays, uint64_t n, uint32_t k, EmuHit* hits, EmuStats* st, uint32_t schedule) {
    static_assert(sizeof(EmuHit) == sizeof(HitX), "one hit record");
    const U4* wide = reinterpret_cast<const U4*>(g_bvh.nodes.data());
    const U4* leaf = g_bvh.leaf.data();
    for (uint64_t i = 0; i < n; ++i) {
        const RayX r = make_ray(rays[i].ox, rays[i].oy, rays[i].oz, rays[i].dx, rays[i].dy, rays[i].dz);
        TravCounters c = { 0, 0, 0, 0, 0, 0, 0 };
        bool overflow = false;
        const uint32_t sched = schedule ? schedule + (uint32_t)i * 2654435761u : 0u;
        trace_wide<HIT_MULTI, true, 256>(wide, leaf, r, rays[i].tmax, &c, &overflow, 0x3F800000u, sched,
                                         reinterpret_cast<HitX*>(hits + i * k), k);
        if (overflow) st->overflow++;
        if (g_emu_stack_overflows) { st->overflow += g_emu_stack_overflows; g_emu_stack_overflows = 0; }
        if (c.max_stack > st->max_stack) st->max_stack = c.max_stack;
        st->wide_visits += c.wide_nodes; st->leaf_blocks += c.leaf_blocks; st->leaf_pass += c.leaf_pass; st->tri_tests += c.tri_tests; st->words += c.words;
    }
}
