// rt_intersect.cuh — ray/sphere tests and closest-hit search (brute-force list and
// flattened BVH).  The sphere tests reproduce the reference's SASS-level operation
// order (nvcc 12.9, sm_100, disassembled from the unchanged src/main.cu):
//   oc    = FADD.RZ                                  (vec3 operator-, vec3.h:272-284)
//   a,b,. = FMUL.RZ products, FADD(RN) sums          (vec3::dot, vec3.h:208-219)
//   c     = FFMA(-r, r, dot(oc,oc))                  (sphere.h:96: ptxas fuses `- _r*_r`)
//   delta = FFMA(b, b, -(FMUL a*c))                  (sphere.h:97)
//   sqrt.rn, div.rn for the roots                    (sphere.h:106-107)
// so that (id, t) of every closest hit is bit-identical to the reference kernel.
#pragma once

#include <float.h>

#include "rt_device.cuh"

namespace rtd {

struct RayQ { // ray + per-ray invariants hoisted out of the primitive loop
    V3 o, d;
    float time;
    float a; // dot(d, d) — recomputed per sphere by the reference (sphere.h:94), same value
};

RT_DEV RayQ make_rayq(const Ray& r) {
    RayQ q;
    q.o = r.o;
    q.d = r.d;
    q.time = r.time;
    q.a = dot(r.d, r.d);
    return q;
}

// sphere::hit (sphere.h:86-140) root selection for closest-hit use.  Returns the
// accepted root (near root if >= tmin, else far root if >= tmin; bounds inclusive) or
// NaN-free "no hit".  The `root > tmax` tests of the reference are subsumed by the
// caller's strict `t < closest` (hitable_list.h:72, bvh.h:147), see DESIGN.md.
RT_DEV bool sphere_root_static(const RayQ& q, float4 s, float tmin, float& t) {
    V3 oc = q.o - mk(s.x, s.y, s.z);
    float b = dot(oc, q.d);
    float c = __fmaf_rn(-s.w, s.w, dot(oc, oc));
    float delta = __fmaf_rn(b, b, -__fmul_rn(q.a, c));
    if (!(delta >= 0.f)) return false; // sphere.h:99 (`delta < 0`), NaN never survives `t < closest`
    float sq = __fsqrt_rn(delta);
    float root = __fdiv_rn(__fadd_rn(-b, -sq), q.a);
    if (root < tmin) {
        root = __fdiv_rn(__fadd_rn(-b, sq), q.a);
        if (root < tmin) return false;
    }
    t = root;
    return true;
}

// moving_sphere::center (sphere.h:49-52): c0 + ((time - t0) / (t1 - t0)) * (c1 - c0)
RT_DEV V3 moving_center(float4 a, float4 b, float dt, float time) {
    float s = __fdiv_rn(__fsub_rn(time, b.w), dt);
    return mk(a.x, a.y, a.z) + s * mk(b.x, b.y, b.z);
}

// moving_sphere::hit (sphere.h:157-190): delta > 0 strictly, roots exclusive of tmin
RT_DEV bool sphere_root_moving(const RayQ& q, float4 a, float4 bq, float dt, float tmin, float& t) {
    V3 oc = q.o - moving_center(a, bq, dt, q.time);
    float b = dot(oc, q.d);
    float c = __fmaf_rn(-a.w, a.w, dot(oc, oc));
    float delta = __fmaf_rn(b, b, -__fmul_rn(q.a, c));
    if (!(delta > 0.f)) return false;
    float sq = __fsqrt_rn(delta);
    float root = __fdiv_rn(__fadd_rn(-b, -sq), q.a);
    if (!(root > tmin)) {
        root = __fdiv_rn(__fadd_rn(-b, sq), q.a);
        if (!(root > tmin)) return false;
    }
    t = root;
    return true;
}

// Closest-hit bookkeeping: strictly smaller t wins (hitable_list.h:72); an exact tie
// goes to the object that comes first in the caller's list, which is what the
// reference's first-found-wins loop does.
RT_DEV void consider(const DScene& sc, uint32_t prim, float t, Hit& best) {
    if (t < best.t) {
        best.t = t;
        best.prim = prim;
    } else if (t == best.t && best.prim != RT_INVALID_ID) {
        if (__ldg(&sc.sph_c[prim]).w < __ldg(&sc.sph_c[best.prim]).w) best.prim = prim;
    }
}

RT_DEV void test_prim(const DScene& sc, const RayQ& q, uint32_t prim, float tmin, Hit& best) {
    float t;
    float4 a = __ldg(&sc.sph_a[prim]);
    if (prim < sc.n_static) {
        if (sphere_root_static(q, a, tmin, t)) consider(sc, prim, t, best);
    } else {
        float4 b = __ldg(&sc.sph_b[prim]);
        float dt = __uint_as_float(__ldg(&sc.sph_c[prim]).x);
        if (sphere_root_moving(q, a, b, dt, tmin, t)) consider(sc, prim, t, best);
    }
}

// hitable_list::hit with bvh == nullptr (hitable_list.h:66-78).  FORM: 0 = decide at run time (the parity hooks and the
// megakernel), 1 = the constant-bank list only, 2 = the global-memory list only — the wavefront kernel of list scenes is
// instantiated for the form its scene uses, so the other loop is not in its instruction stream (the C1 kernel's time follows
// its code size: L1.5 instruction cache = 32 KB).
template <int FORM = 0>
RT_DEV Hit closest_hit_list(const DScene& sc, const RayQ& q, float tmin) {
    Hit best{FLT_MAX, RT_INVALID_ID};
    float t;
    if (FORM == 1 || (FORM == 0 && sc.n_list != 0u)) { // small scene: sphere data from the kernel parameters (constant bank, uniform loads)
        // (rolled on purpose: unrolled over the compile-time index the sphere data become immediate constant operands,
        // but the kernel grows from 3 800 to 5 200 instructions and loses more to instruction-cache misses than the
        // loop control costs — C1 8.01 ms unrolled, 7.41 ms rolled, 7.74 ms with the global-memory list, 8.47 ms round 1;
        // profiles/r02_c1_instruction_diet.md)
#pragma unroll 1
        for (uint32_t i = 0; i < sc.n_static; ++i) {
            if (sphere_root_static(q, sc.lst_a[i], tmin, t)) consider(sc, i, t, best);
        }
#pragma unroll 1
        for (uint32_t i = sc.n_static; i < sc.n_spheres; ++i) {
            if (sphere_root_moving(q, sc.lst_a[i], sc.lst_b[i], sc.lst_dt[i], tmin, t)) consider(sc, i, t, best);
        }
        return best;
    }
    if constexpr (FORM != 1) {
        // two spheres per trip: the second sphere's load is in flight while the first is tested
#pragma unroll 2
        for (uint32_t i = 0; i < sc.n_static; ++i) {
            float4 a = __ldg(&sc.sph_a[i]);
            if (sphere_root_static(q, a, tmin, t)) consider(sc, i, t, best);
        }
        for (uint32_t i = sc.n_static; i < sc.n_spheres; ++i) {
            float4 a = __ldg(&sc.sph_a[i]);
            float4 b = __ldg(&sc.sph_b[i]);
            float dt = __uint_as_float(__ldg(&sc.sph_c[i]).x);
            if (sphere_root_moving(q, a, b, dt, tmin, t)) consider(sc, i, t, best);
        }
    }
    return best;
}

// Conservative slab test.  t = lo * (1/d) - o * (1/d) as one FFMA per bound against the per-ray products
// noi = -(o * 1/d) (12 FFMA for the two boxes of a node instead of 12 FADD + 12 FMUL).  The product o * 1/d is rounded
// once per ray, so every bound carries an extra absolute error of at most 2^-24 * max_k |o_k / d_k| over the
// subtract-then-multiply form; the acceptance test is widened by `e` = 2^-22 * that maximum (and, as before, the far
// bound by 2 ulp), so rounding can only add node visits, never remove a leaf the sphere test would accept (the
// primitive boxes are padded on top of this: rt_bvh_host.cpp sphere_box / k_prim_boxes).
// RT_SLAB_FAR_WIDEN: the far bound (box exit, or the closest t so far) is widened by 2^-8 relative.  The closest-t
// culling must tolerate the NOISE of the reference's sphere arithmetic: at distance D from the ray origin the float
// quadratic (sphere.h:94-107) resolves t only to about 2^-11 * D (dot(oc,oc) - r*r cancels), so a sphere can report a
// t slightly outside the span of its own box.  With the margin the closest hit does not depend on the order in which
// leaves are visited (per-lane loop, speculative rounds, refilled lanes: same image), at 0.4 % more box overlap.
#define RT_SLAB_FAR_WIDEN 1.00390625f
RT_DEV bool slab(float4 lo, float4 hi, const V3& inv, const V3& noi, float e, float tmin, float tmax, float& tnear) {
    float tx0 = __fmaf_rn(lo.x, inv.x, noi.x), tx1 = __fmaf_rn(hi.x, inv.x, noi.x);
    float ty0 = __fmaf_rn(lo.y, inv.y, noi.y), ty1 = __fmaf_rn(hi.y, inv.y, noi.y);
    float tz0 = __fmaf_rn(lo.z, inv.z, noi.z), tz1 = __fmaf_rn(hi.z, inv.z, noi.z);
    float tn = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), tmin));
    float tf = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), tmax));
    tnear = tn;
    return tn <= __fmaf_rn(tf, RT_SLAB_FAR_WIDEN, e);
}

// The same test on a box given as centre c and half-extent h (BvhNodeCH): tm = c * (1/d) - o * (1/d) is the ray parameter at
// the box's centre plane, entry and exit lie half * |1/d| before and behind it — no ordering of two bounds per axis.
// Rounding: tm carries the error of the min/max form's bounds (one FFMA on the per-ray products, covered by `e` and the box
// padding), the second FFMA adds at most 2^-24 of the larger bound — against an acceptance test that is 2^-8 wide.
RT_DEV bool slab_ch(float4 c, float4 h, const V3& inv, const V3& noi, float e, float tmin, float tmax, float& tnear) {
    const float tmx = __fmaf_rn(c.x, inv.x, noi.x), tmy = __fmaf_rn(c.y, inv.y, noi.y), tmz = __fmaf_rn(c.z, inv.z, noi.z);
    const float ax = fabsf(inv.x), ay = fabsf(inv.y), az = fabsf(inv.z);
    const float tn = fmaxf(fmaxf(__fmaf_rn(-h.x, ax, tmx), __fmaf_rn(-h.y, ay, tmy)), fmaxf(__fmaf_rn(-h.z, az, tmz), tmin));
    const float tf = fminf(fminf(__fmaf_rn(h.x, ax, tmx), __fmaf_rn(h.y, ay, tmy)), fminf(__fmaf_rn(h.z, az, tmz), tmax));
    tnear = tn;
    return tn <= __fmaf_rn(tf, RT_SLAB_FAR_WIDEN, e);
}

#define RT_BVH_STACK RT_BVH_STACK_DEPTH
// A 4-wide node is a binary node with its inner children replaced by their children, so a path from the root through a
// tree of binary depth d meets at most ceil(d / 2) 4-wide nodes, and each pushes at most 3 of its 4 children.  A push
// the stack has no room for would drop a subtree (and possibly the closest hit) without any error.
#define RT_BVH4_STACK (3 * ((RT_BVH_STACK_DEPTH + 1) / 2))
static_assert(RT_BVH_STACK_DEPTH != 64 || RT_BVH4_STACK == 96, "depth <= 64: at most 32 4-wide nodes on a path, each pushing at most 3 entries");

// Flattened-BVH closest hit: short per-thread stack, both child boxes fetched with four
// float4 read-only loads per visited node, near child first, culled by the closest t so far.
// (Reference: bvh_node::dfs, bvh.h:121-155 — pointer-chasing, unordered, never culls by
// `closest`, recomputes 1/d for every box: aabb.h:54-68.)
// Resumable traversal state: the persistent wavefront kernel interleaves the traversals of a warp's lanes with
// refilling finished lanes, so the loop body is exposed as two steps.
#define RT_TRAV_DONE 0x7fffffff
struct Trav {
    int node; // >= 0 inner node, < 0 leaf ~prim, RT_TRAV_DONE finished
    int leaf; // speculative traversal: postponed leaf (< 0), or >= 0 for none
    int sp;
    Hit best;
    V3 inv; // 1/d; an axis the ray does not move along (1/d not finite) gets +-2^100: its bounds stay exact (see trav_begin)
    V3 noi; // -(o * inv)
    float e; // widening of the slab acceptance test, 2^-22 * max |o * inv|
};
RT_DEV void trav_begin(const DScene& sc, const RayQ& q, Trav& t) {
    t.node = int(sc.root);
    t.leaf = 0;
    t.sp = 0;
    t.best = Hit{FLT_MAX, RT_INVALID_ID};
    // Per axis: inv = 1/d, noi = -(o * inv).  d == 0 (or so small that 1/d overflows): inv = +-2^100, a power of two, so
    // o * inv is exact and fma(lo, inv, noi) is the correctly rounded (lo - o) * 2^100 — sign-exact like the infinities
    // of the textbook slab test, and without a contribution to `e`.
    const float dk[3] = {q.d.x, q.d.y, q.d.z}, ok[3] = {q.o.x, q.o.y, q.o.z};
    float iv[3], no[3], m = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        iv[k] = 1.0f / dk[k];
        if (fabsf(iv[k]) <= 3.0e38f) {
            no[k] = -(ok[k] * iv[k]);
            m = fmaxf(m, fabsf(no[k]));
        } else {
            iv[k] = copysignf(1.2676506e30f, dk[k]); // 2^100
            no[k] = -(ok[k] * iv[k]);
        }
    }
    t.inv = V3{iv[0], iv[1], iv[2]};
    t.noi = V3{no[0], no[1], no[2]};
    t.e = m * 2.3841858e-7f; // 2^-22
}
// One visit of a binary node (BvhNodeCH; precondition: t.node >= 0 && t.node != RT_TRAV_DONE).
// (lmin / lmax / rmin / rmax: centre and half-extent of the left, then of the right child)
RT_DEV void trav_inner(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    const float4* np = reinterpret_cast<const float4*>(sc.nodes_ch + t.node);
    float4 lmin = __ldg(np + 0), lmax = __ldg(np + 1), rmin = __ldg(np + 2), rmax = __ldg(np + 3);
    float tl, tr;
    const bool hl = slab_ch(lmin, lmax, t.inv, t.noi, t.e, tmin, t.best.t, tl);
    const bool hr = slab_ch(rmin, rmax, t.inv, t.noi, t.e, tmin, t.best.t, tr);
    const int cl = __float_as_int(lmin.w), cr = __float_as_int(lmax.w);
    if (hl && hr) {
        const bool left_first = tl <= tr;
        if (t.sp < RT_BVH_STACK) stack[t.sp++] = left_first ? cr : cl;
        t.node = left_first ? cl : cr;
    } else if (hl) {
        t.node = cl;
    } else if (hr) {
        t.node = cr;
    } else {
        t.node = t.sp ? stack[--t.sp] : RT_TRAV_DONE;
    }
}
// The end of every 4-wide node visit: the `nhit` hit children (key = entry distance, +inf for a miss) ordered with a
// 5-comparator network; the nearest is walked next, the others are pushed farthest first.
RT_DEV void trav_next4(Trav& t, int* stack, float (&key)[4], int (&ref)[4], int nhit) {
#define RT_CSWAP(a, b)                       \
    {                                        \
        const bool sw = key[b] < key[a];     \
        const float ka = key[a], kb = key[b]; \
        const int ra = ref[a], rb = ref[b];  \
        key[a] = sw ? kb : ka;               \
        key[b] = sw ? ka : kb;               \
        ref[a] = sw ? rb : ra;               \
        ref[b] = sw ? ra : rb;               \
    }
    RT_CSWAP(0, 1) RT_CSWAP(2, 3) RT_CSWAP(0, 2) RT_CSWAP(1, 3) RT_CSWAP(1, 2)
#undef RT_CSWAP
    if (nhit > 3 && t.sp < RT_BVH4_STACK) stack[t.sp++] = ref[3];
    if (nhit > 2 && t.sp < RT_BVH4_STACK) stack[t.sp++] = ref[2];
    if (nhit > 1 && t.sp < RT_BVH4_STACK) stack[t.sp++] = ref[1];
    // (requesting the second-nearest child into L1 with prefetch.global.L1 while the nearest is walked: C4 1 487 -> 1 420 Mrays/s,
    // profiles/r02_c4_ab_travq.log — the kernel is short of load slots, not of hits)
    t.node = nhit ? ref[0] : (t.sp ? stack[--t.sp] : RT_TRAV_DONE);
}
// One visit of a 128-byte 4-wide node (BvhNode4): seven vector loads, four slab tests in SoA form, then trav_next4.
RT_DEV void trav_inner4(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    const float4* np = reinterpret_cast<const float4*>(sc.nodes4 + t.node);
    const float4 mnx = __ldg(np + 0), mny = __ldg(np + 1), mnz = __ldg(np + 2);
    const float4 mxx = __ldg(np + 3), mxy = __ldg(np + 4), mxz = __ldg(np + 5);
    const int4 refs = __ldg(reinterpret_cast<const int4*>(np + 6));
    float key[4];
    int ref[4] = {refs.x, refs.y, refs.z, refs.w};
    const float lox[4] = {mnx.x, mnx.y, mnx.z, mnx.w}, loy[4] = {mny.x, mny.y, mny.z, mny.w}, loz[4] = {mnz.x, mnz.y, mnz.z, mnz.w};
    const float hix[4] = {mxx.x, mxx.y, mxx.z, mxx.w}, hiy[4] = {mxy.x, mxy.y, mxy.z, mxy.w}, hiz[4] = {mxz.x, mxz.y, mxz.z, mxz.w};
    int nhit = 0;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        float tn;
        const bool hit = slab(make_float4(lox[s], loy[s], loz[s], 0.f), make_float4(hix[s], hiy[s], hiz[s], 0.f), t.inv, t.noi, t.e, tmin,
                              t.best.t, tn) && ref[s] != RT_BVH4_EMPTY;
        key[s] = hit ? tn : __int_as_float(0x7f800000); // +inf: misses sort to the end
        nhit += hit ? 1 : 0;
    }
    trav_next4(t, stack, key, ref, nhit);
}
// One visit of a QUANTISED 4-wide node (BvhNode4Q): four 16-byte loads instead of seven.  The ray is moved into the
// node's grid once per axis — s = unit * (1/d), o = p * (1/d) - origin * (1/d), the same FFMA form as slab() — and every
// bound is then ONE FFMA on a byte: t = q * s + o.  The decoded boxes contain the float boxes with a whole unit to
// spare (k_quantize4), so the test can only add visits; acceptance test, far-bound margin, ordering network and stack
// discipline are those of the 128-byte form.
// three-input minimum / maximum (FMNMX3, sm_100)
RT_DEV float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
RT_DEV float fmin3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
// byte K of `w` as the float 1 + byte * 2^-15: ONE byte permute (ALU pipe) drops it into the mantissa of 1.0f
template <int K>
RT_DEV float byte_m(uint32_t w) { return __uint_as_float(__byte_perm(w, 0x3F800000u, 0x7604u | (uint32_t(K) << 4))); }
RT_DEV void trav_inner_q(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    const uint4* np = reinterpret_cast<const uint4*>(sc.nodes4q + t.node);
    const uint4 q0 = __ldg(np + 0), q1 = __ldg(np + 1), q2 = __ldg(np + 2), q3 = __ldg(np + 3);
    // 2^15 units per axis (the exponent bytes are at most 20 + 127)
    const float Sx = __uint_as_float(((q0.w & 0xffu) << 23) + (15u << 23)) * t.inv.x;
    const float Sy = __uint_as_float(((q0.w & 0xff00u) << 15) + (15u << 23)) * t.inv.y;
    const float Sz = __uint_as_float(((q0.w & 0xff0000u) << 7) + (15u << 23)) * t.inv.z;
    const float ox = __fmaf_rn(__uint_as_float(q0.x), t.inv.x, t.noi.x);
    const float oy = __fmaf_rn(__uint_as_float(q0.y), t.inv.y, t.noi.y);
    const float oz = __fmaf_rn(__uint_as_float(q0.z), t.inv.z, t.noi.z);
    float key[4];
    int ref[4] = {int(q1.x), int(q1.y), int(q1.z), int(q1.w)};
    int nhit = 0;
    // The sign of 1/d says which face of a box the ray enters through, for all four children at once: the word of entry
    // bytes and the word of exit bytes are selected per axis (6 selects per node) instead of ordering two bounds per axis
    // and child (24 min/max).  With the byte in the mantissa — 1 + b * 2^-15 — the bound is t = f * S + O with
    // S = 2^15 * s and O = o - S; O is rounded at the magnitude of the node's own extent, 2^-9 of a unit below the whole
    // unit the quantised boxes have to spare (k_quantize4), so the test still only adds visits.
    const float Ox = ox - Sx, Oy = oy - Sy, Oz = oz - Sz;
    const bool px = t.inv.x >= 0.f, py = t.inv.y >= 0.f, pz = t.inv.z >= 0.f;
    const uint32_t nx = px ? q2.x : q2.w, fx = px ? q2.w : q2.x;
    const uint32_t ny = py ? q2.y : q3.x, fy = py ? q3.x : q2.y;
    const uint32_t nz = pz ? q2.z : q3.y, fz = pz ? q3.y : q2.z;
    const float far_max = t.best.t;
#define RT_CHILD(S)                                                                                                               \
    {                                                                                                                             \
        const float tn = fmax3(__fmaf_rn(byte_m<S>(nx), Sx, Ox), __fmaf_rn(byte_m<S>(ny), Sy, Oy),                                \
                               fmaxf(__fmaf_rn(byte_m<S>(nz), Sz, Oz), tmin));                                                    \
        const float tf = fmin3(__fmaf_rn(byte_m<S>(fx), Sx, Ox), __fmaf_rn(byte_m<S>(fy), Sy, Oy),                                \
                               fminf(__fmaf_rn(byte_m<S>(fz), Sz, Oz), far_max));                                                 \
        const bool hit = tn <= __fmaf_rn(tf, RT_SLAB_FAR_WIDEN, t.e) && ref[S] != RT_BVH4_EMPTY;                                  \
        key[S] = hit ? tn : __int_as_float(0x7f800000); /* +inf: misses sort to the end */                                       \
        nhit += hit ? 1 : 0;                                                                                                      \
    }
    RT_CHILD(0) RT_CHILD(1) RT_CHILD(2) RT_CHILD(3)
#undef RT_CHILD
    trav_next4(t, stack, key, ref, nhit);
}
// one leaf test (precondition: t.node < 0)
RT_DEV void trav_leaf(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    test_prim(sc, q, uint32_t(~t.node), tmin, t.best);
    t.node = t.sp ? stack[--t.sp] : RT_TRAV_DONE;
}

RT_DEV Hit closest_hit_bvh(const DScene& sc, const RayQ& q, float tmin) {
    int stack[RT_BVH_STACK];
    Trav t;
    trav_begin(sc, q, t);
    // "while-while" traversal: leaves travel through `node` and the stack like inner nodes, so the lanes of a
    // warp first all descend through inner nodes and then test their pending leaves together, instead of each
    // lane stopping for a sphere test in the middle of the others' descent.
    while (true) {
        while (t.node >= 0 && t.node != RT_TRAV_DONE) trav_inner(sc, q, tmin, t, stack);
        if (t.node == RT_TRAV_DONE) break;
        trav_leaf(sc, q, tmin, t, stack);
    }
    return t.best;
}

// The same walk over the 4-wide nodes (the tree k_wf_step_pt traverses; built from RT_PT_MIN_SPHERES primitives on):
// per-lane loop, used by the parity hook (rt_trace_primary, use_bvh = 2) so that the wide traversal is compared
// with the reference kernel ray by ray.
template <bool QUANT = false>
RT_DEV Hit closest_hit_bvh4(const DScene& sc, const RayQ& q, float tmin) {
    int stack[RT_BVH4_STACK];
    Trav t;
    trav_begin(sc, q, t);
    t.node = int(sc.root4);
    while (true) {
        while (t.node >= 0 && t.node != RT_TRAV_DONE) {
            if (QUANT) trav_inner_q(sc, q, tmin, t, stack);
            else trav_inner4(sc, q, tmin, t, stack);
        }
        if (t.node == RT_TRAV_DONE) break;
        trav_leaf(sc, q, tmin, t, stack);
    }
    return t.best;
}

// Warp-cooperative variant for kernels that reach the traversal with all 32 lanes converged (the wavefront step
// kernels): speculative while-while traversal (Aila & Laine 2009).  A lane that reaches a leaf does not stop and
// wait for the other lanes' descents — it postpones the leaf and keeps walking inner nodes until every lane of the
// warp holds a leaf (or has nothing left); then all pending leaves are tested together.  The postponed leaf cannot
// shorten the ray while it waits, so a few extra nodes are visited, but the result is the same (closest t, ties to
// the lower list ordinal: order-independent).  ncu on C4 (1 M spheres, one sphere per leaf): the plain per-lane
// loop above ran with 5 of 32 lanes active because every lane waited at every leaf for the longest inner run.
// MUST be called by all 32 lanes of the warp; lanes without a ray pass has_ray = false.
RT_DEV void trav_inner_spec(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    trav_inner(sc, q, tmin, t, stack);
    if (t.node < 0 && t.leaf >= 0) { // first leaf: postpone it, go on with the next node
        t.leaf = t.node;
        t.node = t.sp ? stack[--t.sp] : RT_TRAV_DONE;
    }
}
// one warp round: inner nodes until no lane is still looking for a leaf, then the pending leaves
RT_DEV void trav_round_warp(const DScene& sc, const RayQ& q, float tmin, Trav& t, int* stack) {
    for (;;) {
        const bool inner = t.node >= 0 && t.node != RT_TRAV_DONE;
        if (!__any_sync(0xffffffffu, inner && t.leaf >= 0)) break;
        if (inner) trav_inner_spec(sc, q, tmin, t, stack);
    }
    while (t.leaf < 0) {
        test_prim(sc, q, uint32_t(~t.leaf), tmin, t.best);
        t.leaf = 0;
        if (t.node < 0) { // the node after the postponed leaf is a leaf too
            t.leaf = t.node;
            t.node = t.sp ? stack[--t.sp] : RT_TRAV_DONE;
        }
    }
}
RT_DEV Hit closest_hit_bvh_warp(const DScene& sc, const RayQ& q, float tmin, bool has_ray) {
    int stack[RT_BVH_STACK];
    Trav t;
    trav_begin(sc, q, t);
    if (!has_ray) t.node = RT_TRAV_DONE;
    while (__any_sync(0xffffffffu, t.node != RT_TRAV_DONE)) trav_round_warp(sc, q, tmin, t, stack);
    return t.best;
}

RT_DEV Hit closest_hit(const DScene& sc, const RayQ& q, float tmin, bool use_bvh) {
    return (use_bvh && sc.nodes) ? closest_hit_bvh(sc, q, tmin) : closest_hit_list(sc, q, tmin);
}

// Surface data of an accepted hit: p = o + t*d (ray.h:28-30), outward normal
// n = (p - c)/r (sphere.h:123), both in the reference's RZ arithmetic.
RT_DEV void hit_surface(const DScene& sc, const RayQ& q, Hit h, V3& p, V3& n) {
    float4 a = __ldg(&sc.sph_a[h.prim]);
    V3 c = mk(a.x, a.y, a.z);
    if (h.prim >= sc.n_static) {
        float4 b = __ldg(&sc.sph_b[h.prim]);
        float dt = __uint_as_float(__ldg(&sc.sph_c[h.prim]).x);
        c = moving_center(a, b, dt, q.time);
    }
    p = q.o + h.t * q.d;
    n = (p - c) / a.w;
}

// sphere::get_sphere_uv (sphere.h:61-83): atan2f/asinf in float, the affine map in double.
// KAT (sphere.h:71-77): (1,0,0)->(.5,.5) (0,1,0)->(.5,1) (0,0,1)->(.25,.5) (-1,0,0)->(0,.5)
RT_DEV void sphere_uv(V3 n, float& u, float& v) {
    float phi = atan2f(n.z, n.x);
    float theta = asinf(n.y);
    u = 1 - (phi + 3.14159265358979323846) / (2 * 3.14159265358979323846);
    v = (theta + 1.57079632679489661923) / 3.14159265358979323846;
}

} // namespace rtd
