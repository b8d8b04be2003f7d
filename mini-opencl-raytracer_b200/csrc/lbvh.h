// lbvh.h -- device-side binary BVH build (lbvh.cu): Morton sort + Karras hierarchy + bottom-up refit over primitive
// groups, flattened on the device into the reference's CLLinearBVHNode array and triangle order.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include "b2rt_types.h"

namespace b2rt {

// Scratch bytes lbvh_build needs for m groups.
size_t lbvh_scratch_bytes(uint32_t m);

// d_group_bounds: m x {min.xyz, max.xyz}; d_first: m + 1 first-triangle indices of the groups (loader order). Outputs
// (device): the 2m - 1 nodes in the REFERENCE's format and order (CLLinearBVHNode, pre-order, first child at index + 1,
// `offset` = second child or first triangle) and d_order[k] = loader index of the triangle that becomes triangle k. m >= 2.
cudaError_t lbvh_build(const float* d_group_bounds, const uint32_t* d_first, uint32_t m, const float scene_lo[3], const float scene_hi[3],
                       void* d_scratch, RefNode* d_nodes, uint32_t* d_order, uint64_t* launches, cudaStream_t st);

// Exclusive scan of m uint32 values on `st` (d_in and d_out must not overlap). d_sums: scan_scratch_words(m) words; on return d_sums[0]
// holds the total.
size_t scan_scratch_words(uint32_t m);
cudaError_t scan_exclusive(const uint32_t* d_in, uint32_t m, uint32_t* d_out, uint32_t* d_sums, uint64_t* launches, cudaStream_t st);

}  // namespace b2rt
