// rt_lbvh.cu — GPU LBVH build for large scenes (BASELINE.json north_star (1)): motion-union
// AABBs -> 63-bit Morton codes of the box centres -> radix sort -> Karras' parallel binary
// radix tree -> bottom-up refit, written straight into the flattened 64-byte two-child-box
// node array the traversal kernel reads (rt_device.cuh BvhNode).  Replaces the reference's
// single-thread recursive median split with an in-thread sort per level (bvh.h:75-113),
// which is O(N log^2 N) on one GPU thread and cannot build 10^6 primitives in useful time.
#include "rt_lbvh.cuh"
#include "rt_kernels.cuh"

#include <utility>

#include "rt_prims.cuh"

namespace rtd {

namespace {

__device__ __forceinline__ unsigned flip_f(float f) { // order-preserving float -> uint
    unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float unflip_f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// Bounds of primitive `prim` (sphere.h:142-146; moving: union of the boxes at both ends of the motion, sphere.h:192-202),
// padded exactly like the host builder (rt_bvh_host.cpp sphere_box) so the conservative slab test never rejects a ray the
// rounded sphere test accepts.  The LBVH build (k_prim_boxes) and the refit of a resident tree (k_refit_all) both use it.
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

// Primitive bounds (prim_box) and their centroid bounds.
__global__ void __launch_bounds__(256) k_prim_boxes(const float4* __restrict__ sph_a, const float4* __restrict__ sph_b,
                                                    const uint32_t* __restrict__ ids, uint32_t n, uint32_t n_static,
                                                    float4* __restrict__ lo, float4* __restrict__ hi,
                                                    unsigned* __restrict__ cbounds) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float c[3] = {0.f, 0.f, 0.f};
    bool valid = i < n;
    if (valid) {
        const uint32_t prim = ids ? ids[i] : i;
        float l[3], h[3];
        prim_box(sph_a, sph_b, prim, n_static, l, h);
#pragma unroll
        for (int k = 0; k < 3; ++k) c[k] = 0.5f * l[k] + 0.5f * h[k];
        lo[i] = make_float4(l[0], l[1], l[2], 0.f);
        hi[i] = make_float4(h[0], h[1], h[2], 0.f);
    }
    // centroid bounds: warp reduce, then one atomic per warp and axis
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        unsigned mn = valid ? flip_f(c[k]) : 0xffffffffu, mx = valid ? flip_f(c[k]) : 0u;
        mn = __reduce_min_sync(0xffffffffu, mn);
        mx = __reduce_max_sync(0xffffffffu, mx);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&cbounds[k], mn);
            atomicMax(&cbounds[3 + k], mx);
        }
    }
}

__device__ __forceinline__ unsigned long long spread21(unsigned long long x) { // 21 bits -> every third bit
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void __launch_bounds__(256) k_morton(const float4* __restrict__ lo, const float4* __restrict__ hi, uint32_t n,
                                                const unsigned* __restrict__ cbounds, unsigned long long* __restrict__ keys,
                                                uint32_t* __restrict__ vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 l = lo[i], h = hi[i];
    float c[3] = {0.5f * l.x + 0.5f * h.x, 0.5f * l.y + 0.5f * h.y, 0.5f * l.z + 0.5f * h.z};
    // one scale for all axes (the largest extent): Morton cells are cubes, so a flat scene is split along its long
    // axes first instead of being cut into thin layers
    float ext = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) ext = fmaxf(ext, unflip_f(cbounds[3 + k]) - unflip_f(cbounds[k]));
    unsigned long long code = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float mn = unflip_f(cbounds[k]);
        float t = ext > 0.f ? (c[k] - mn) / ext : 0.f;
        unsigned long long q = (unsigned long long)fminf(fmaxf(t * 2097152.f, 0.f), 2097151.f);
        code |= spread21(q) << (2 - k);
    }
    keys[i] = code;
    vals[i] = i;
}

// Karras 2012: length of the common prefix of keys i and j; ties are broken by the index so
// duplicate codes still form a proper tree.
__device__ __forceinline__ int delta(const unsigned long long* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(unsigned(i) ^ unsigned(j));
    return __clzll(a ^ b);
}

// One thread per internal node: range, split, children.  Node 0 is the root.
__global__ void __launch_bounds__(256) k_topology(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                  const uint32_t* __restrict__ ids, int n, BvhNode* __restrict__ nodes,
                                                  int* __restrict__ parent_inner, int* __restrict__ parent_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = (delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) >> 1;; t = (t + 1) >> 1) {
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    int gamma = i + s * d + min(d, 0);
    int lo_ = min(i, j), hi_ = max(i, j);
    int left, right;
    if (lo_ == gamma) {
        left = ~int(ids ? ids[vals[gamma]] : vals[gamma]);
        parent_leaf[gamma] = i;
    } else {
        left = gamma;
        parent_inner[gamma] = i;
    }
    if (hi_ == gamma + 1) {
        right = ~int(ids ? ids[vals[gamma + 1]] : vals[gamma + 1]);
        parent_leaf[gamma + 1] = i;
    } else {
        right = gamma + 1;
        parent_inner[gamma + 1] = i;
    }
    // boxes are filled by the refit; only the child references are written here
    reinterpret_cast<int*>(&nodes[i].lmin)[3] = left;
    reinterpret_cast<int*>(&nodes[i].lmax)[3] = right;
    if (i == 0) parent_inner[0] = -1;
}

// One thread per leaf climbs towards the root.  A thread writes its subtree's box into its
// side of the parent node; the first thread to reach a node stops, the second (which then sees
// both child boxes) carries the union upwards.
__global__ void __launch_bounds__(256) k_refit(const uint32_t* __restrict__ vals, const uint32_t* __restrict__ ids, int n,
                                               const float4* __restrict__ lo, const float4* __restrict__ hi, BvhNode* nodes,
                                               const int* __restrict__ parent_inner, const int* __restrict__ parent_leaf,
                                               unsigned* __restrict__ visits, float* __restrict__ root_box) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint32_t ci = vals[k]; // compact index of the primitive: lo/hi are indexed by it
    float4 bl = lo[ci], bh = hi[ci];
    int me = ~int(ids ? ids[ci] : ci);
    int parent = parent_leaf[k];
    while (parent >= 0) {
        if (!refit_step(nodes, parent, me, bl, bh, visits)) return;
        me = parent;
        parent = parent_inner[parent];
    }
    // only the thread that closed the root gets here: (bl, bh) bound the whole tree
    root_box[0] = bl.x; root_box[1] = bl.y; root_box[2] = bl.z;
    root_box[3] = bh.x; root_box[4] = bh.y; root_box[5] = bh.z;
}

// depth of the deepest leaf (for the traversal stack bound): every leaf walks its parent chain
__global__ void __launch_bounds__(256) k_depth(int n, const int* __restrict__ parent_inner, const int* __restrict__ parent_leaf,
                                               unsigned* __restrict__ max_depth) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned d = 0;
    if (k < n) {
        int p = parent_leaf[k];
        while (p >= 0) {
            ++d;
            p = parent_inner[p];
        }
    }
    d = __reduce_max_sync(0xffffffffu, d);
    if ((threadIdx.x & 31) == 0) atomicMax(max_depth, d);
}

// The parent table of a binary node array (host SAH tree, LBVH, and the chain of outsized spheres above the LBVH root alike:
// one primitive per leaf, child < 0 is leaf ~prim): parent_inner[i] for every node, parent_leaf[p] for every primitive.
// Both are -1 before this kernel; the root keeps -1.
__global__ void __launch_bounds__(256) k_parents(const BvhNode* __restrict__ nodes, uint32_t n_nodes, int* __restrict__ parent_inner,
                                                 int* __restrict__ parent_leaf) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const float4* np = reinterpret_cast<const float4*>(nodes + i);
    const int child[2] = {__float_as_int(np[0].w), __float_as_int(np[1].w)};
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        if (child[c] >= 0) parent_inner[child[c]] = int(i);
        else parent_leaf[~child[c]] = int(i);
    }
}

// One thread per primitive: its padded box (prim_box, as the builders pad it), then up the tree with the visit-counter
// protocol of the LBVH build's k_refit.  Every node is written on both sides, so no box of the old tree survives.
__global__ void __launch_bounds__(256) k_refit_all(const float4* __restrict__ sph_a, const float4* __restrict__ sph_b, uint32_t n,
                                                   uint32_t n_static, BvhNode* nodes, const int* __restrict__ parent_inner,
                                                   const int* __restrict__ parent_leaf, unsigned* __restrict__ visits) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    float l[3], h[3];
    prim_box(sph_a, sph_b, k, n_static, l, h);
    float4 bl = make_float4(l[0], l[1], l[2], 0.f), bh = make_float4(h[0], h[1], h[2], 0.f);
    int me = ~int(k);
    for (int parent = parent_leaf[k]; parent >= 0; parent = parent_inner[parent]) {
        if (!refit_step(nodes, parent, me, bl, bh, visits)) return;
        me = parent;
    }
}

// Binary -> 4-wide: node i of the 4-wide array is binary node i with each inner child replaced by that child's two
// children.  Every binary node is converted (one thread each, no topology walk); a traversal that starts at the root
// only ever reaches the nodes two binary levels apart.
__global__ void __launch_bounds__(256) k_collapse4(const BvhNode* __restrict__ nodes, uint32_t n_nodes, BvhNode4* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const float4* np = reinterpret_cast<const float4*>(nodes + i);
    const float4 lmin = np[0], lmax = np[1], rmin = np[2], rmax = np[3];
    float lo[4][3], hi[4][3];
    int ref[4];
    int k = 0;
    auto put = [&](int r, float4 a, float4 b) {
        lo[k][0] = a.x; lo[k][1] = a.y; lo[k][2] = a.z;
        hi[k][0] = b.x; hi[k][1] = b.y; hi[k][2] = b.z;
        ref[k++] = r;
    };
    const int child[2] = {__float_as_int(lmin.w), __float_as_int(lmax.w)};
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        if (child[c] >= 0) {
            const float4* cp = reinterpret_cast<const float4*>(nodes + child[c]);
            const float4 a = cp[0], b = cp[1], cc = cp[2], d = cp[3];
            put(__float_as_int(a.w), a, b);
            put(__float_as_int(b.w), cc, d);
        } else {
            put(child[c], c ? rmin : lmin, c ? rmax : lmax);
        }
    }
    for (; k < 4;) put(RT_BVH4_EMPTY, make_float4(0.f, 0.f, 0.f, 0.f), make_float4(0.f, 0.f, 0.f, 0.f));
    BvhNode4 o;
    o.mnx = make_float4(lo[0][0], lo[1][0], lo[2][0], lo[3][0]);
    o.mny = make_float4(lo[0][1], lo[1][1], lo[2][1], lo[3][1]);
    o.mnz = make_float4(lo[0][2], lo[1][2], lo[2][2], lo[3][2]);
    o.mxx = make_float4(hi[0][0], hi[1][0], hi[2][0], hi[3][0]);
    o.mxy = make_float4(hi[0][1], hi[1][1], hi[2][1], hi[3][1]);
    o.mxz = make_float4(hi[0][2], hi[1][2], hi[2][2], hi[3][2]);
    o.refs = make_int4(ref[0], ref[1], ref[2], ref[3]);
    o.pad = make_int4(0, 0, 0, 0);
    out[i] = o;
}

} // namespace

namespace {
// nodes a walk from the root can reach in the 4-wide graph, level by level (level[i] = distance from the root + 1)
__global__ void __launch_bounds__(256) k_mark4(const BvhNode4* __restrict__ n4, uint32_t n_nodes, uint32_t* __restrict__ level, uint32_t cur) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes || level[i] != cur) return;
    const int4 r = n4[i].refs;
    const int ref[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (ref[k] >= 0 && ref[k] != RT_BVH4_EMPTY) level[ref[k]] = cur + 1u;
}
__global__ void __launch_bounds__(256) k_used4(const uint32_t* __restrict__ level, uint32_t n_nodes, uint32_t* __restrict__ used) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_nodes) used[i] = level[i] ? 1u : 0u;
}
__global__ void __launch_bounds__(256) k_compact4(const BvhNode4* __restrict__ in, const uint32_t* __restrict__ level,
                                                  const uint32_t* __restrict__ idx, uint32_t n_nodes, BvhNode4* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes || level[i] == 0u) return;
    BvhNode4 n = in[i];
    int* r = reinterpret_cast<int*>(&n.refs);
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (r[k] >= 0 && r[k] != RT_BVH4_EMPTY) r[k] = int(idx[r[k]]);
    out[idx[i]] = n;
}
} // namespace

namespace {
// 64-byte form of the dense 4-wide nodes (BvhNode4Q, rt_device.cuh).  Per axis: unit = the smallest power of two with
// extent / unit <= 251 (and >= 4 ulp of the coordinates, so that the corner's own rounding stays inside the margin),
// corner p = min - unit rounded DOWN, lo byte = floor((lo - p) / unit) - 1 >= 0, hi byte = ceil((hi - p) / unit) + 1 <= 255:
// every decoded bound lies at least one unit outside the float box.  Nodes this cannot represent (units beyond 2^20,
// a clamped byte) raise `bad`; the scene then keeps the 128-byte nodes.
__global__ void __launch_bounds__(256) k_quantize4(const BvhNode4* __restrict__ in, uint32_t n, BvhNode4Q* __restrict__ out,
                                                   uint32_t* __restrict__ bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const BvhNode4 nd = in[i];
    const float lo[3][4] = {{nd.mnx.x, nd.mnx.y, nd.mnx.z, nd.mnx.w}, {nd.mny.x, nd.mny.y, nd.mny.z, nd.mny.w}, {nd.mnz.x, nd.mnz.y, nd.mnz.z, nd.mnz.w}};
    const float hi[3][4] = {{nd.mxx.x, nd.mxx.y, nd.mxx.z, nd.mxx.w}, {nd.mxy.x, nd.mxy.y, nd.mxy.z, nd.mxy.w}, {nd.mxz.x, nd.mxz.y, nd.mxz.z, nd.mxz.w}};
    const int ref[4] = {nd.refs.x, nd.refs.y, nd.refs.z, nd.refs.w};
    uint32_t qlo[3] = {0u, 0u, 0u}, qhi[3] = {0u, 0u, 0u}, exps = 0u;
    float p[3];
    bool ok = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        double mn = 1e300, mx = -1e300;
        for (int c = 0; c < 4; ++c)
            if (ref[c] != RT_BVH4_EMPTY) {
                mn = fmin(mn, double(lo[a][c]));
                mx = fmax(mx, double(hi[a][c]));
            }
        if (mn > mx) mn = mx = 0.0;
        int e = -100;
        if (mx > mn) {
            frexp((mx - mn) / 251.0, &e); // (mx - mn) / 251 = m * 2^e with m in [0.5, 1): 2^e >= (mx - mn) / 251
        }
        const double mag = fmax(fabs(mn), fabs(mx));
        if (mag > 0.0) {
            int em;
            frexp(mag, &em);        // mag < 2^em: ulp(mag) <= 2^(em - 24)
            e = max(e, em - 24 + 2); // unit >= 4 ulp of the coordinates
        }
        e = max(e, -100);
        ok = ok && e <= 20 && isfinite(mn) && isfinite(mx);
        e = min(e, 20);
        const double unit = ldexp(1.0, e);
        const float pa = __double2float_rd(mn - unit);
        p[a] = pa;
        exps |= uint32_t(e + 127) << (8 * a);
        for (int c = 0; c < 4; ++c) {
            uint32_t bl = 255u, bh = 0u; // an empty slot: inverted box (and its reference says so)
            if (ref[c] != RT_BVH4_EMPTY) {
                const double l = floor((double(lo[a][c]) - double(pa)) / unit) - 1.0;
                const double h = ceil((double(hi[a][c]) - double(pa)) / unit) + 1.0;
                ok = ok && l >= 0.0 && h <= 255.0;
                bl = uint32_t(fmin(fmax(l, 0.0), 255.0));
                bh = uint32_t(fmin(fmax(h, 0.0), 255.0));
            }
            qlo[a] |= bl << (8 * c);
            qhi[a] |= bh << (8 * c);
        }
    }
    if (!ok) atomicOr(bad, 1u);
    BvhNode4Q q;
    q.q0 = make_uint4(__float_as_uint(p[0]), __float_as_uint(p[1]), __float_as_uint(p[2]), exps);
    q.q1 = make_uint4(uint32_t(ref[0]), uint32_t(ref[1]), uint32_t(ref[2]), uint32_t(ref[3]));
    q.q2 = make_uint4(qlo[0], qlo[1], qlo[2], qhi[0]);
    q.q3 = make_uint4(qhi[1], qhi[2], 0u, 0u);
    out[i] = q;
}
} // namespace

namespace {
// one box: centre rounded to nearest, half-extent = the larger of the two distances from THAT centre to the bounds, rounded up
__device__ __forceinline__ void box_ch(float lo, float hi, float& c, float& h) {
    c = __fadd_rn(__fmul_rn(0.5f, lo), __fmul_rn(0.5f, hi));
    h = fmaxf(__fsub_ru(hi, c), __fsub_ru(c, lo));
    if (!(h >= 0.f)) h = 0.f; // (an inverted / NaN box stays empty)
}
__global__ void __launch_bounds__(256) k_nodes_ch(const BvhNode* __restrict__ in, uint32_t n, BvhNodeCH* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const BvhNode nd = in[i];
    BvhNodeCH o;
    o.lmin.w = nd.lmin.w; // left child
    o.lmax.w = nd.lmax.w; // right child
    o.rmin.w = o.rmax.w = 0.f;
    box_ch(nd.lmin.x, nd.lmax.x, o.lmin.x, o.lmax.x);
    box_ch(nd.lmin.y, nd.lmax.y, o.lmin.y, o.lmax.y);
    box_ch(nd.lmin.z, nd.lmax.z, o.lmin.z, o.lmax.z);
    box_ch(nd.rmin.x, nd.rmax.x, o.rmin.x, o.rmax.x);
    box_ch(nd.rmin.y, nd.rmax.y, o.rmin.y, o.rmax.y);
    box_ch(nd.rmin.z, nd.rmax.z, o.rmin.z, o.rmax.z);
    out[i] = o;
}
} // namespace
cudaError_t bvh_nodes_ch(const BvhNode* nodes, uint32_t n, BvhNodeCH* out, cudaStream_t st) {
    if (n) k_nodes_ch<<<(n + 255) / 256, 256, 0, st>>>(nodes, n, out);
    return cudaGetLastError();
}

// out_q (may be nullptr) receives the quantised form of the first *n_out nodes of `out`; *quant_ok tells whether every node
// was representable.
cudaError_t bvh_quantize4(const BvhNode4* nodes4, uint32_t n4, BvhNode4Q* out_q, bool* quant_ok, cudaStream_t st) {
    *quant_ok = false;
    if (n4 == 0 || !out_q) return cudaSuccess;
    PoolBuffer<uint32_t> bad;
    cudaError_t e = bad.alloc(1, st);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(bad.get(), 0, sizeof(uint32_t), st);
    if (e == cudaSuccess) {
        k_quantize4<<<(n4 + 255) / 256, 256, 0, st>>>(nodes4, n4, out_q, bad.get());
        e = cudaGetLastError();
    }
    uint32_t h = 1u;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&h, bad.get(), sizeof h, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    *quant_ok = e == cudaSuccess && h == 0u;
    return e;
}

// 4-wide form of a finished binary tree.  Only every other level of the binary tree survives as a 4-wide node, so
// the reachable nodes are marked from the root, numbered by an exclusive scan and written densely: the array a ray
// walks is then as large as the binary one (n/2 nodes of 128 B) and can be pinned in L2 as a whole.
cudaError_t bvh_collapse4(const BvhNode* nodes, uint32_t n_nodes, uint32_t root, uint32_t depth, BvhNode4* out, uint32_t* n_out,
                          uint32_t* root_out, cudaStream_t st) {
    *n_out = 0;
    *root_out = 0;
    if (n_nodes == 0) return cudaSuccess;
    PoolBuffer<BvhNode4> wide;
    PoolBuffer<uint32_t> level, used, idx, tmp;
    RTD_TRY(wide.alloc(n_nodes, st));
    RTD_TRY(level.alloc(size_t(n_nodes) + 1, st));
    RTD_TRY(used.alloc(size_t(n_nodes) + 1, st));
    RTD_TRY(idx.alloc(size_t(n_nodes) + 1, st));
    RTD_TRY(tmp.alloc(prims::scan_scratch_elems(size_t(n_nodes) + 1), st));
    const unsigned blocks = (n_nodes + 255) / 256;
    k_collapse4<<<blocks, 256, 0, st>>>(nodes, n_nodes, wide.get());
    RTD_TRY(cudaMemsetAsync(level.get(), 0, size_t(n_nodes + 1) * sizeof(uint32_t), st));
    const uint32_t one = 1u;
    RTD_TRY(cudaMemcpyAsync(level.get() + root, &one, sizeof one, cudaMemcpyHostToDevice, st));
    for (uint32_t cur = 1; cur <= depth / 2 + 2; ++cur) k_mark4<<<blocks, 256, 0, st>>>(wide.get(), n_nodes, level.get(), cur);
    k_used4<<<(n_nodes + 256) / 256, 256, 0, st>>>(level.get(), n_nodes + 1, used.get()); // level[n_nodes] == 0: the scan's total slot
    RTD_TRY(prims::exclusive_sum<uint32_t>(used.get(), idx.get(), size_t(n_nodes) + 1, tmp.get(), st));
    k_compact4<<<blocks, 256, 0, st>>>(wide.get(), level.get(), idx.get(), n_nodes, out);
    RTD_TRY(cudaGetLastError());
    uint32_t h[2] = {0, 0};
    RTD_TRY(cudaMemcpyAsync(&h[0], idx.get() + n_nodes, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RTD_TRY(cudaMemcpyAsync(&h[1], idx.get() + root, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RTD_TRY(cudaStreamSynchronize(st));
    *n_out = h[0];
    *root_out = h[1];
    return cudaSuccess;
}

// The scratch is stream-ordered pool memory (the context keeps freed blocks): no device-wide synchronisation per scene build.
cudaError_t lbvh_build(const float4* sph_a, const float4* sph_b, uint32_t n_static, const uint32_t* ids, uint32_t n,
                       BvhNode* nodes, cudaStream_t st, float* ms, uint32_t* depth, float root_box[6]) {
    if (n < 2) return cudaErrorInvalidValue;
    PoolBuffer<float4> lo, hi;
    PoolBuffer<unsigned long long> keys_a, keys_b;
    PoolBuffer<uint32_t> vals_a, vals_b, tmp;
    PoolBuffer<int> parent_inner, parent_leaf;
    PoolBuffer<unsigned> visits, scal; // scal: [0..5] centroid bounds, [6] depth, [8..13] root box
    TimingEvent e0, e1;
    RTD_TRY(lo.alloc(n, st));
    RTD_TRY(hi.alloc(n, st));
    RTD_TRY(keys_a.alloc(n, st));
    RTD_TRY(keys_b.alloc(n, st));
    RTD_TRY(vals_a.alloc(n, st));
    RTD_TRY(vals_b.alloc(n, st));
    RTD_TRY(parent_inner.alloc(n, st));
    RTD_TRY(parent_leaf.alloc(n, st));
    RTD_TRY(visits.alloc(n, st));
    RTD_TRY(scal.alloc(16, st));
    RTD_TRY(tmp.alloc(prims::sort_scratch_elems(n), st));
    RTD_TRY(e0.create());
    RTD_TRY(e1.create());

    const unsigned init[8] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u, 0u, 0u};
    RTD_TRY(cudaMemcpyAsync(scal.get(), init, sizeof init, cudaMemcpyHostToDevice, st));
    RTD_TRY(cudaEventRecord(e0.ev, st));
    RTD_TRY(cudaMemsetAsync(visits.get(), 0, n * sizeof(unsigned), st));
    const unsigned blocks = (n + 255) / 256;
    unsigned long long *keys = keys_a.get(), *keys_out = keys_b.get();
    uint32_t *vals = vals_a.get(), *vals_out = vals_b.get();
    k_prim_boxes<<<blocks, 256, 0, st>>>(sph_a, sph_b, ids, n, n_static, lo.get(), hi.get(), scal.get());
    k_morton<<<blocks, 256, 0, st>>>(lo.get(), hi.get(), n, scal.get(), keys, vals);
    { // stable LSD radix sort of the (63-bit Morton code, primitive) pairs: 8 passes of 8 bits (rt_prims.cuh)
        bool in_alt = false;
        RTD_TRY(prims::sort_pairs_u64_u32(keys, vals, keys_out, vals_out, n, 8, tmp.get(), &in_alt, st));
        if (!in_alt) { // the sorted pairs are in (keys, vals): the code below reads (keys_out, vals_out)
            std::swap(keys, keys_out);
            std::swap(vals, vals_out);
        }
    }
    k_topology<<<blocks, 256, 0, st>>>(keys_out, vals_out, ids, int(n), nodes, parent_inner.get(), parent_leaf.get());
    k_refit<<<blocks, 256, 0, st>>>(vals_out, ids, int(n), lo.get(), hi.get(), nodes, parent_inner.get(), parent_leaf.get(),
                                    visits.get(), reinterpret_cast<float*>(scal.get() + 8));
    k_depth<<<blocks, 256, 0, st>>>(int(n), parent_inner.get(), parent_leaf.get(), scal.get() + 6);
    RTD_TRY(cudaEventRecord(e1.ev, st));
    RTD_TRY(cudaGetLastError());
    unsigned d = 0;
    float rb[6] = {0, 0, 0, 0, 0, 0};
    RTD_TRY(cudaMemcpyAsync(&d, scal.get() + 6, sizeof d, cudaMemcpyDeviceToHost, st));
    RTD_TRY(cudaMemcpyAsync(rb, scal.get() + 8, sizeof rb, cudaMemcpyDeviceToHost, st));
    RTD_TRY(cudaStreamSynchronize(st));
    if (root_box)
        for (int k = 0; k < 6; ++k) root_box[k] = rb[k];
    if (ms) RTD_TRY(cudaEventElapsedTime(ms, e0.ev, e1.ev));
    if (depth) *depth = d;
    return cudaSuccess;
}

cudaError_t bvh_parents(const BvhNode* nodes, uint32_t n_nodes, uint32_t n_prims, int* parents, uint32_t* levels, cudaStream_t st) {
    PoolBuffer<unsigned> d_levels;
    RTD_TRY(d_levels.alloc(1, st));
    RTD_TRY(cudaMemsetAsync(parents, 0xff, (size_t(n_nodes) + n_prims) * sizeof(int), st));
    RTD_TRY(cudaMemsetAsync(d_levels.get(), 0, sizeof(unsigned), st));
    k_parents<<<(n_nodes + 255) / 256, 256, 0, st>>>(nodes, n_nodes, parents, parents + n_nodes);
    k_depth<<<(n_prims + 255) / 256, 256, 0, st>>>(int(n_prims), parents, parents + n_nodes, d_levels.get());
    RTD_TRY(cudaGetLastError());
    RTD_TRY(cudaMemcpyAsync(levels, d_levels.get(), sizeof *levels, cudaMemcpyDeviceToHost, st));
    return cudaStreamSynchronize(st);
}

cudaError_t bvh_refit(const float4* sph_a, const float4* sph_b, uint32_t n, uint32_t n_static, BvhNode* nodes, uint32_t n_nodes,
                      const int* parents, cudaStream_t st) {
    PoolBuffer<unsigned> visits;
    RTD_TRY(visits.alloc(n_nodes, st));
    RTD_TRY(cudaMemsetAsync(visits.get(), 0, n_nodes * sizeof(unsigned), st));
    k_refit_all<<<(n + 255) / 256, 256, 0, st>>>(sph_a, sph_b, n, n_static, nodes, parents, parents + n_nodes, visits.get());
    return cudaGetLastError();
}

} // namespace rtd
