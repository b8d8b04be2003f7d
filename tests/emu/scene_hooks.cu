// scene_hooks.cu -- test-only view into a b2rt_context: copies the compressed wide BVH a handle derived (wide nodes, leaf
// blocks, shading records, child_bin, leaf_dir) and its stack bound to the host, so that the device derivation
// (b2rt_build_scene_device) can be compared with the host derivation (b2rt_upload_scene) byte for byte. Built by
// __graft_entry__.build() into tests/emu/libscenehooks.so; the product never links it.
#include <cuda_runtime.h>
#include <string.h>
#include "context.h"

// Sizes in bytes: sizes[0..4] = wide nodes, leaf blocks, shading records, child_bin, leaf_dir. Call once with null
// outputs to learn them (the scene must have been derived: b2rt_scene_info_get first). 0 on success.
extern "C" int b2rt_test_derived_arrays(b2rt_context* ctx, unsigned long long sizes[5], void* wide, void* leaf, void* shade, void* child_bin,
                                        void* leaf_dir, unsigned* stack_bound) {
    if (!ctx || ctx->scene_dirty || !ctx->d_wide) return 1;
    sizes[0] = ctx->info.wide_node_bytes;
    sizes[1] = ctx->info.leaf_bytes;
    sizes[2] = ctx->info.shading_bytes;
    sizes[3] = ctx->info.n_wide_nodes * 32ull;
    sizes[4] = ctx->info.n_leaf_blocks * 8ull;
    if (stack_bound) *stack_bound = ctx->stack_bound;
    if (!wide) return 0;
    if (cudaSetDevice(ctx->device) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) return 2;
    const void* src[5] = { ctx->d_wide, ctx->d_leaf, ctx->d_shade, ctx->d_child_bin, ctx->d_leaf_dir };
    void* dst[5] = { wide, leaf, shade, child_bin, leaf_dir };
    for (int i = 0; i < 5; ++i)
        if (sizes[i] && cudaMemcpy(dst[i], src[i], sizes[i], cudaMemcpyDeviceToHost) != cudaSuccess) return 3;
    return 0;
}
