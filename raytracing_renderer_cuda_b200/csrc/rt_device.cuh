// rt_device.cuh — device-side POD scene, reference-faithful vector arithmetic and
// the counter-based RNG shared by every kernel of the render path.
//
// Arithmetic convention (SURVEY.md §8a "Q17"): the reference's vec3 operators are
// explicit round-toward-zero intrinsics on the device (vec3.h:73-151,258-347), so
// nothing inside vector math is FMA-contracted; dot()/sq_length() are RZ multiplies
// summed left-to-right with round-to-nearest adds (vec3.h:168-179,208-219).  The
// geometric part of this renderer (intersection, hit point, normal, scattered ray)
// reproduces those roundings with the same intrinsics so closest-hit results are
// bit-identical to the reference kernel; colour math is ordinary FP32.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rt_api.h"
#include "rt_fastdiv.hpp"

namespace rtd {

#define RT_DEV __device__ __forceinline__

// ---------------------------------------------------------------- vec3 (RZ) ----
struct V3 {
    float x, y, z;
};
RT_DEV V3 mk(float x, float y, float z) { return V3{x, y, z}; }
RT_DEV V3 operator+(V3 a, V3 b) { return V3{__fadd_rz(a.x, b.x), __fadd_rz(a.y, b.y), __fadd_rz(a.z, b.z)}; }
RT_DEV V3 operator-(V3 a, V3 b) { return V3{__fsub_rz(a.x, b.x), __fsub_rz(a.y, b.y), __fsub_rz(a.z, b.z)}; }
RT_DEV V3 operator*(V3 a, V3 b) { return V3{__fmul_rz(a.x, b.x), __fmul_rz(a.y, b.y), __fmul_rz(a.z, b.z)}; }
RT_DEV V3 operator*(V3 a, float t) { return V3{__fmul_rz(a.x, t), __fmul_rz(a.y, t), __fmul_rz(a.z, t)}; }
RT_DEV V3 operator*(float t, V3 a) { return V3{__fmul_rz(a.x, t), __fmul_rz(a.y, t), __fmul_rz(a.z, t)}; }
// __fdiv_rz / __fsqrt_rz, bit for bit, without the out-of-line subroutine ptxas emits for the .rz forms (div.rz.f32: a
// CALL into ~66 instructions of exponent juggling per quotient; ncu on C1: the three quotients of n = (p - c) / r were
// 12 % of all instructions a shaded hit executes, profiles/r02_c1_instruction_diet.md).  The round-to-NEAREST forms have
// an inline fast path; the correctly rounded nearest result q is either the truncated one or one ulp beyond it, and ONE
// exact FMA residual tells which: q*y - x (resp. s*s - x) is computed exactly before its single rounding, so its sign
// is exact, and it has the sign of x (is positive) exactly when q (s) was rounded away from zero.  Stepping the bit
// pattern down by one then gives the truncated result — also from +-inf to +-FLT_MAX when the quotient overflows, as
// div.rz does.  NaN and x/0 fall through unchanged (every comparison with the NaN residual is false).  Operands so small
// that the residual itself could underflow to zero take the library path.
RT_DEV float div_rz(float x, float y) {
    if (!(fabsf(x) >= 8.6736174e-19f)) return __fdiv_rz(x, y); // |x| < 2^-60 (or NaN): rare, exact by construction
    const float q = __fdiv_rn(x, y);
    const float rem = __fmaf_rn(q, y, -x);
    const bool away = (x > 0.f && rem > 0.f) || (x < 0.f && rem < 0.f);
    return away ? __int_as_float(__float_as_int(q) - 1) : q;
}
RT_DEV float sqrt_rz(float x) {
    if (!(x >= 8.6736174e-19f)) return __fsqrt_rz(x); // tiny, zero, negative, NaN
    const float s = __fsqrt_rn(x);
    const float rem = __fmaf_rn(s, s, -x);
    return rem > 0.f ? __int_as_float(__float_as_int(s) - 1) : s;
}
// vec3 / float (vec3.h:334-347).  Inline: one out-of-line copy per kernel is 350 instructions smaller but its call spills
// around every use (C1 8.07 ms against 7.43 ms inline; profiles/r02_c1_instruction_diet.md).
RT_DEV V3 operator/(V3 a, float t) { return V3{div_rz(a.x, t), div_rz(a.y, t), div_rz(a.z, t)}; }
RT_DEV V3 operator-(V3 a) { return V3{-a.x, -a.y, -a.z}; }
// vec3::dot (vec3.h:208-219): RZ products, RN sums, left to right
RT_DEV float dot(V3 a, V3 b) {
    return __fadd_rn(__fadd_rn(__fmul_rz(a.x, b.x), __fmul_rz(a.y, b.y)), __fmul_rz(a.z, b.z));
}
RT_DEV float length(V3 a) { return sqrt_rz(dot(a, a)); } // vec3.h:153-166
RT_DEV V3 normalize(V3 a) {                                  // vec3.h:199-205
    if (a.x == 0.f && a.y == 0.f && a.z == 0.f) return a;
    return a / length(a);
}

// ---------------------------------------------------------------- scene PODs ----
struct DCamera { // camera.h:40-47, filled on the host by rt_scene_create
    V3 origin, lower_left, horizontal, vertical, u, v;
    float lens_radius, t0, t1;
};

struct DMaterial { // 32 B, read as 2 x float4
    uint32_t kind;
    int32_t tex;
    float ax, ay, az; // metal albedo / dielectric tint
    float param;      // roughness / ri / intensity
    float pad0, pad1;
};

struct DTexture { // 48 B, read as 3 x float4
    uint32_t kind;
    int32_t even, odd, image;
    float c1x, c1y, c1z, density;
    float c2x, c2y, c2z, hardness;
};

struct DImage {
    cudaTextureObject_t tex;
    int32_t width, height;
};

// 64-byte BVH node holding the boxes of BOTH children, so one node visit is four
// float4 read-only loads and decides both subtrees.  child >= 0: inner node index;
// child < 0: leaf, primitive index = ~child (one sphere per leaf).
struct BvhNode {
    float4 lmin; // (L.min.xyz, as_float(left child))
    float4 lmax; // (L.max.xyz, as_float(right child))
    float4 rmin; // (R.min.xyz, unused)
    float4 rmax; // (R.max.xyz, unused)
};

// The binary node as the traversal reads it (round 2): every child box as CENTRE and HALF-EXTENT,
//   (L.centre.xyz, as_float(left child)), (L.half.xyz, as_float(right child)), (R.centre.xyz, -), (R.half.xyz, -),
// written by k_nodes_ch (rt_lbvh.cu) from the min/max node with the half-extent rounded UP, so that
// [centre - half, centre + half] contains the min/max box.  The slab test then needs no ordering of two bounds per axis:
// entry = tm - half * |1/d|, exit = tm + half * |1/d| with tm = centre * (1/d) - o * (1/d) — three FFMA per axis
// instead of two FFMA and two FMNMX (the ALU pipe is the busiest one of the BVH kernels: 58 % on C2).
typedef BvhNode BvhNodeCH;

// 128-byte 4-wide node: the two children of a binary node replaced by their own children (a leaf child stays).
// Slot s: box (mn?.s, mx?.s), reference refs.s (>= 0 inner node — the index of the BINARY node it was made from —,
// < 0 leaf ~prim, RT_BVH4_EMPTY unused).  Built from the binary array by k_collapse4 (rt_lbvh.cu).
struct BvhNode4 {
    float4 mnx, mny, mnz, mxx, mxy, mxz;
    int4 refs;
    int4 pad;
};
#define RT_BVH4_EMPTY 0x7fffffff

// The same 4-wide node in 64 bytes (round 2): the child boxes as 8-bit offsets from the node's own corner, in units of a
// per-axis power of two — decoded box = p + q * 2^e, at least one unit OUTSIDE the float box on every side (k_quantize4,
// rt_lbvh.cu), so the walk stays conservative and the closest hit is unchanged (leaves test the spheres themselves).
// Why: ncu on the 1 M-sphere scene showed k_wf_step_pt bound by L1 request slots, not by latency alone (l1tex 88 % busy:
// every lane fetches its own 128-byte node with seven LDG.128, one tag look-up each); four loads per visit instead of seven.
//   q0 = (p.x, p.y, p.z, ex | ey << 8 | ez << 16)   e? = biased exponent byte of the unit (float bits = e? << 23)
//   q1 = refs[4]
//   q2 = (lo.x[4], lo.y[4], lo.z[4], hi.x[4])       one byte per child
//   q3 = (hi.y[4], hi.z[4], 0, 0)
struct BvhNode4Q {
    uint4 q0, q1, q2, q3;
};

#define RT_MAX_IMAGES 8
#define RT_LIST_MAX 12 // scenes of up to this many spheres travel inside the kernel parameters (constant bank), see DScene::lst_*
// Deepest binary tree a scene may have (rt_scene_create rejects deeper ones).  The binary walks push at most one entry per
// inner ancestor, so this is also their stack size; the 4-wide walks need RT_BVH4_STACK entries (rt_intersect.cuh).
#define RT_BVH_STACK_DEPTH 64

struct DScene {
    // primitives, static spheres first: [0, n_static) static, [n_static, n) moving
    const float4* sph_a;  // (c0.xyz, r)
    const float4* sph_b;  // (rz(c1-c0).xyz, t0)       — moving spheres only
    const uint4* sph_c;   // (as_uint(t1-t0), material, id, ordinal in the caller's list)
    uint32_t n_spheres;
    uint32_t n_static;
    const BvhNode* nodes; // nullptr => brute force
    const BvhNode4* nodes4; // 4-wide form of the same tree (densely renumbered), nullptr if not built
    const BvhNodeCH* nodes_ch; // the binary nodes in centre / half-extent form (same numbering): what trav_inner reads
    const BvhNode4Q* nodes4q; // ... and its 64-byte quantised form (same numbering), nullptr if not built / not representable
    uint32_t n_nodes4;
    uint32_t root4;
    uint32_t n_nodes;
    uint32_t root;        // index of the BVH root node
    const DMaterial* mats;
    const DTexture* texs;
    uint32_t has_noise;   // any Perlin-based texture (noise / wood): the kernels stage the permutation table
    DImage images[RT_MAX_IMAGES];
    DCamera cam;
    uint32_t n_lights;              // emitter spheres (RT_RENDER_EMITTER_SAMPLING), at most RT_MAX_LIGHTS
    uint32_t lights[RT_MAX_LIGHTS]; // their primitive indices, in the caller's list order
    // Brute-force list scenes (n_spheres <= RT_LIST_MAX, no BVH — C1's 8 spheres, the hdr scene's 3): a copy of sph_a /
    // sph_b / dt inside the kernel parameters.  The list loop's index is warp-uniform, so the sphere data are read from
    // the constant bank through the uniform datapath (LDCU) instead of one LDG.128 + 64-bit address arithmetic per
    // sphere and ray (ncu, C1: those and the loop control were 5 % of the kernel's instructions).  n_list = 0: not filled.
    uint32_t n_list;
    float4 lst_a[RT_LIST_MAX]; // (c0.xyz, r)
    float4 lst_b[RT_LIST_MAX]; // (rz(c1 - c0).xyz, t0)
    float lst_dt[RT_LIST_MAX]; // t1 - t0
};

struct DRenderParams {
    FastDiv div_width; // pixel -> (column, row)
    FastDiv div_npix;  // path -> (sample, pixel), see PathMap
    int32_t width, height;
    int32_t spp, sample_offset;
    int32_t max_depth;
    uint32_t seed;
    float tmin;
    float world_r, world_g, world_b;
    float bloom;
    uint32_t flags; // RT_RENDER_*
    // Adaptive sampling (the ADAPT instantiations of the render kernels; nullptr / 0 otherwise): path x of a pass is pixel
    // adapt_pixels[x mod n] of sample sample_offset + x / n with n = div_npix.d, and a finished path adds into plane
    // (sample - adapt_first) & 1 of a two-plane accumulator whose planes are adapt_plane float4 apart (rt_adaptive.cu).
    const uint32_t* adapt_pixels;
    uint32_t adapt_first;
    uint32_t adapt_plane;
    // Frame sequences (the FRAMES instantiations; nullptr otherwise): spp counts the samples of the whole batch, n_frames
    // times div_spp.d per pixel.  Sample s belongs to frame f = (s - sample_offset) / div_spp.d, whose camera is
    // frame_cams[f] and whose accumulator is the f-th width*height block of float4 (rt_api.cu, frames_into).
    const DCamera* frame_cams;
    FastDiv div_spp;
};

// Which paths a render kernel instantiation traces (its RM template argument): every pixel of the frame (RM_PLAIN), the
// pixel list of an adaptive pass (RM_ADAPT), or the frames of a sequence (RM_FRAMES).
enum : int { RM_PLAIN = 0, RM_ADAPT = 1, RM_FRAMES = 2 };

// frame of a sample in FRAMES instantiations (computed at ray generation and at accumulation only, never per bounce)
RT_DEV uint32_t frame_of(const DRenderParams& rp, uint32_t sample) { return fastdiv(sample - uint32_t(rp.sample_offset), rp.div_spp); }

// the float4 accumulator a path of `sample` adds into: the render's own, in ADAPT instantiations the plane of the sample's
// parity, in FRAMES instantiations the sample's frame
template <int RM>
RT_DEV float4* accum_plane(float4* accum, const DRenderParams& rp, uint32_t sample) {
    if (RM == RM_ADAPT) return accum + size_t((sample - rp.adapt_first) & 1u) * rp.adapt_plane;
    if (RM == RM_FRAMES) return accum + size_t(frame_of(rp, sample)) * rp.div_npix.d;
    return accum;
}

struct Ray {
    V3 o, d;
    float time;
};

struct Hit {
    float t;
    uint32_t prim; // index into sph_* (RT_INVALID_ID on miss)
};

// ---------------------------------------------------------------- Philox4x32-10 ----
// Counter-based RNG keyed on (pixel, sample, bounce): the stream a path sees does
// not depend on which thread, kernel or GPU evaluates it.  (The reference carries a
// per-pixel XORWOW state, main.cu:76-95,111 — per-sample parity with it is impossible
// by construction; parity is distributional.)
struct U4 {
    uint32_t x, y, z, w;
};
RT_DEV U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0;
        c1 = lo1;
        c2 = n2;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}
// draw block `blk` of (pixel, sample, bounce); bounce 0 = camera
RT_DEV U4 rng_block(uint32_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, uint32_t blk) {
    return philox4x32_10(pixel, sample, (bounce << 8) | blk, 0x52544232u, seed, 0x42323030u);
}
// curand_uniform's mapping, (0,1]  (reference draws: main.cu:116-117, utils.h:69-72,84-85)
RT_DEV float u01(uint32_t x) { return __fmaf_rn((float)x, 2.3283064365386963e-10f, 1.1641532182693481e-10f); }

// Uniform point in the open unit ball.  The reference rejects points of the cube
// (utils.h:61-77, mean 1.91 tries of 3 uniforms); this draws the same distribution
// directly (uniform direction x cbrt radius) so every lane does the same work.
RT_DEV V3 sample_unit_ball(float u1, float u2, float u3) {
    float z = __fmaf_rn(-2.f, u1, 1.f);
    float rxy = sqrtf(fmaxf(0.f, __fmaf_rn(-z, z, 1.f)));
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    float rad = fminf(cbrtf(u3), 0.99999994f);
    return V3{rad * rxy * c, rad * rxy * s, rad * z};
}
// Uniform point in the open unit disk (reference: rejection, utils.h:79-91)
RT_DEV void sample_unit_disk(float u1, float u2, float& dx, float& dy) {
    float rad = fminf(sqrtf(u1), 0.99999994f);
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    dx = rad * c;
    dy = rad * s;
}

} // namespace rtd
