// rt_lbvh.cuh — GPU LBVH build (Morton codes over the motion-union AABBs -> radix sort ->
// Karras topology -> bottom-up refit) into the flattened 64-byte node array.
#pragma once

#include <cuda_runtime.h>

#include "rt_device.cuh"

namespace rtd {

// sph_a / sph_b: the device sphere arrays of DScene (static spheres first); prim index = array index.
// ids_dev: the m primitives to build over (nullptr: all of [0, m)); m >= 2.  Writes m-1 BvhNode, root = 0.
// ms: device time of the build; depth: deepest leaf; root_box: lo.xyz, hi.xyz of the whole tree (host array).
cudaError_t lbvh_build(const float4* sph_a, const float4* sph_b, uint32_t n_static, const uint32_t* ids_dev, uint32_t m,
                       BvhNode* nodes_dev, cudaStream_t st, float* ms, uint32_t* depth, float root_box[6]);

// 4-wide form of a finished binary node array (host SAH or LBVH, incl. nodes appended above the root)
// out: room for n_nodes entries; n_out: nodes written (the reachable ones, densely numbered); root_out: index of the root
// centre / half-extent form of n binary nodes (BvhNodeCH, rt_device.cuh); conservative: half-extents are rounded up
cudaError_t bvh_nodes_ch(const BvhNode* nodes, uint32_t n, BvhNodeCH* out, cudaStream_t st);
cudaError_t bvh_quantize4(const BvhNode4* nodes4, uint32_t n4, BvhNode4Q* out_q, bool* quant_ok, cudaStream_t st);
cudaError_t bvh_collapse4(const BvhNode* nodes, uint32_t n_nodes, uint32_t root, uint32_t depth, BvhNode4* out, uint32_t* n_out,
                          uint32_t* root_out, cudaStream_t st);

// parent table of a finished binary node array: parents[i] of node i, then parents[n_nodes + p] of primitive p (root: -1);
// levels: the depth of its deepest leaf (synchronises)
cudaError_t bvh_parents(const BvhNode* nodes, uint32_t n_nodes, uint32_t n_prims, int* parents, uint32_t* levels, cudaStream_t st);
// every box of the binary node array from the current primitives, bottom-up along the parent table; the topology stays
cudaError_t bvh_refit(const float4* sph_a, const float4* sph_b, uint32_t n, uint32_t n_static, BvhNode* nodes, uint32_t n_nodes,
                      const int* parents, cudaStream_t st);

} // namespace rtd
