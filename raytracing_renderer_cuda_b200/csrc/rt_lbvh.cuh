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

// Bounds of primitive `prim` (sphere.h:142-146; moving: union of the boxes at both ends of the motion, sphere.h:192-202),
// padded exactly like the host builder (rt_bvh_host.cpp sphere_box) so the conservative slab test never rejects a ray the
// rounded sphere test accepts.  The LBVH build (k_prim_boxes) and the scene update's refit (rt_update.cu) both use it.
__device__ __forceinline__ void prim_box(const float4* __restrict__ sph_a, const float4* __restrict__ sph_b, uint32_t prim,
                                         uint32_t n_static, float l[3], float h[3]) {
    float4 a = __ldg(&sph_a[prim]);
    float c0[3] = {a.x, a.y, a.z}, c1[3] = {a.x, a.y, a.z};
    if (prim >= n_static) {
        float4 b = __ldg(&sph_b[prim]);
        c1[0] = __fadd_rz(a.x, b.x); // where moving_center() puts the sphere at the end of its motion
        c1[1] = __fadd_rz(a.y, b.y);
        c1[2] = __fadd_rz(a.z, b.z);
    }
    float ar = fabsf(a.w);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float lk = fminf(c0[k], c1[k]) - ar, hk = fmaxf(c0[k], c1[k]) + ar;
        float pad = ar * 6.1035156e-5f + (fabsf(lk) + fabsf(hk)) * 3.8146973e-6f;
        l[k] = lk - pad;
        h[k] = hk + pad;
    }
}

// One step of the bottom-up refit, run by one thread per leaf: the thread writes its subtree's box (bl, bh) into its side of
// node `parent` (the side whose child reference is `me`).  The first thread to reach a node returns false; the second, which
// then sees both child boxes, returns true with their union in (bl, bh) and carries it on to the node's parent.
__device__ __forceinline__ bool refit_step(BvhNode* nodes, int parent, int me, float4& bl, float4& bh, unsigned* visits) {
    BvhNode* nd = nodes + parent;
    volatile float* f = reinterpret_cast<volatile float*>(nd);
    int left = reinterpret_cast<const int*>(&nd->lmin)[3];
    if (left == me) {
        f[0] = bl.x; f[1] = bl.y; f[2] = bl.z;
        f[4] = bh.x; f[5] = bh.y; f[6] = bh.z;
    } else {
        f[8] = bl.x; f[9] = bl.y; f[10] = bl.z; f[11] = 0.f;
        f[12] = bh.x; f[13] = bh.y; f[14] = bh.z; f[15] = 0.f;
    }
    __threadfence();
    if (atomicAdd(&visits[parent], 1u) == 0u) return false; // sibling subtree not finished yet
    __threadfence();
    bl = make_float4(fminf(f[0], f[8]), fminf(f[1], f[9]), fminf(f[2], f[10]), 0.f);
    bh = make_float4(fmaxf(f[4], f[12]), fmaxf(f[5], f[13]), fmaxf(f[6], f[14]), 0.f);
    return true;
}

} // namespace rtd
