// rt_scene.cu — a scene's lifetime: rt_scene_create (validation, the packed sphere records, the binary tree, the node forms
// derived from it, materials, textures and image arrays), rt_scene_update (edits of sphere records, material records and the
// camera of a resident scene, and the refit of every node form of its tree on the device), rt_scene_update_device (sphere
// edits read, checked, packed and scattered on the device, then the same refit), rt_scene_get_info and rt_scene_destroy.  An update keeps the tree's topology as it was built; only its boxes change (DESIGN.md "Scene updates").
#include <algorithm>
#include <cfenv>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "rt_bvh_host.hpp"
#include "rt_internal.hpp"
#include "rt_lbvh.cuh"
#include "rt_prims.cuh"

namespace rtd {
namespace {

// dst[idx[j]] = src[j]
template <class T>
__global__ void __launch_bounds__(256) k_scatter(const T* __restrict__ src, const uint32_t* __restrict__ idx, uint32_t n, T* __restrict__ dst) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) dst[idx[j]] = src[j];
}

template <class T>
void launch_scatter(const T* src, const uint32_t* idx, uint32_t n, T* dst, cudaStream_t st) {
    if (n) k_scatter<T><<<(n + 255) / 256, 256, 0, st>>>(src, idx, n, dst);
}

template <class T>
rt_status dev_alloc(rt_scene* s, T** out, size_t count) {
    *out = nullptr;
    if (count == 0) return RT_OK;
    void* p = nullptr;
    CUDA_TRY(cudaMallocFromPoolAsync(&p, count * sizeof(T), s->ctx->pool, s->ctx->stream)); // the context's pool: no map/unmap per scene
    s->allocs.push_back(p);
    s->info.device_bytes += count * sizeof(T);
    *out = static_cast<T*>(p);
    return RT_OK;
}

// (an exponent field below all ones: the same test in host and device code)
__host__ __device__ bool finite1(float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    return (u & 0x7f800000u) != 0x7f800000u;
}
__host__ __device__ bool finite3(const float* v) { return finite1(v[0]) && finite1(v[1]) && finite1(v[2]); }

rt_status check_material(const rt_material& m, uint32_t n_textures) {
    ARG_CHECK(m.kind <= RT_MAT_EMITTER, "bad material kind");
    if (m.kind == RT_MAT_LAMBERTIAN || m.kind == RT_MAT_EMITTER)
        ARG_CHECK(m.texture >= 0 && uint32_t(m.texture) < n_textures, "material texture out of range");
    return RT_OK;
}

// The rules of an edited sphere, in the order they are checked; a description's spheres are checked by the last two.
// One definition for the host checks (check_sphere, check_edit) and the device check of rt_scene_update_device (k_check).
enum SphereRule : uint32_t { SPH_OK, SPH_INDEX_RANGE, SPH_REPEATED, SPH_KIND, SPH_MATERIAL, SPH_NOT_FINITE };
const char* const kSphereRuleMessage[] = {
    "", "sphere index out of range", "sphere index repeated",
    "an edit cannot make a static sphere moving or a moving one static", // (static spheres are stored before the moving ones)
    "sphere material out of range", "sphere centre / radius / time is not finite"};

__host__ __device__ uint32_t sphere_rule(const rt_sphere& sp, uint32_t n_materials) {
    // non-finite geometry would reach the builders' bin arithmetic (undefined for NaN / infinity) and the slab tests
    if (!(sp.material < n_materials)) return SPH_MATERIAL;
    if (!(finite3(sp.center0) && finite3(sp.center1) && finite1(sp.radius) && finite1(sp.time0) && finite1(sp.time1)))
        return SPH_NOT_FINITE;
    return SPH_OK;
}

// sphere `sp` replacing list ordinal `i` of a scene of `n` spheres; `repeated`: an earlier position of the edit holds `i`;
// `stored_moving`: the sphere at `i` is stored as a moving one (both read only when i < n)
__host__ __device__ uint32_t sphere_edit_rule(const rt_sphere& sp, uint32_t i, uint32_t n, bool repeated, bool stored_moving,
                                              uint32_t n_materials) {
    if (i >= n) return SPH_INDEX_RANGE;
    if (repeated) return SPH_REPEATED;
    if (((sp.flags & RT_SPHERE_MOVING) != 0) != stored_moving) return SPH_KIND;
    return sphere_rule(sp, n_materials);
}

rt_status check_sphere(const rt_sphere& sp, uint32_t n_materials) {
    const uint32_t r = sphere_rule(sp, n_materials);
    ARG_CHECK(r == SPH_OK, kSphereRuleMessage[r]);
    return RT_OK;
}

// depth[i] = the checker levels above the leaves of texture i (0 for a leaf), by one depth-first walk over every texture
// (children already checked in range).  The stack holds the path being walked, so a child on it closes a cycle.
rt_status checker_depths(const rt_texture* t, uint32_t n, std::vector<uint32_t>& depth) {
    enum : uint8_t { NEW, ON_PATH, DONE };
    std::vector<uint8_t> state(n, NEW);
    std::vector<uint32_t> path;
    depth.assign(n, 0);
    for (uint32_t root = 0; root < n; ++root) {
        if (state[root] != NEW) continue;
        path.push_back(root);
        while (!path.empty()) {
            const uint32_t i = path.back();
            state[i] = ON_PATH;
            if (t[i].kind == RT_TEX_CHECKER) {
                const uint32_t even = uint32_t(t[i].even), odd = uint32_t(t[i].odd);
                if (state[even] == ON_PATH || state[odd] == ON_PATH) {
                    set_error("invalid argument: checker texture %u is its own descendant (a checker cycle)", i);
                    return RT_ERR_INVALID_ARG;
                }
                if (state[even] == NEW || state[odd] == NEW) {
                    path.push_back(state[even] == NEW ? even : odd);
                    continue;
                }
                depth[i] = 1 + std::max(depth[even], depth[odd]);
            }
            state[i] = DONE;
            path.pop_back();
        }
    }
    return RT_OK;
}

rt_status validate_desc(const rt_scene_desc* d) {
    ARG_CHECK(d != nullptr, "desc is NULL");
    ARG_CHECK(d->n_spheres == 0 || d->spheres, "spheres is NULL");
    ARG_CHECK(d->n_materials == 0 || d->materials, "materials is NULL");
    ARG_CHECK(d->n_textures == 0 || d->textures, "textures is NULL");
    ARG_CHECK(d->n_images == 0 || d->images, "images is NULL");
    ARG_CHECK(d->n_images <= RT_MAX_IMAGES, "too many images (max 8)");
    ARG_CHECK(d->bvh_mode <= RT_BVH_GPU_LBVH, "bad bvh_mode");
    for (uint32_t i = 0; i < d->n_images; ++i)
        ARG_CHECK(d->images[i].rgb && d->images[i].width > 0 && d->images[i].height > 0, "empty image");
    for (uint32_t i = 0; i < d->n_textures; ++i) {
        const rt_texture& t = d->textures[i];
        ARG_CHECK(t.kind <= RT_TEX_IMAGE, "bad texture kind");
        if (t.kind == RT_TEX_CHECKER)
            ARG_CHECK(t.even >= 0 && uint32_t(t.even) < d->n_textures && t.odd >= 0 && uint32_t(t.odd) < d->n_textures,
                      "checker child out of range");
        if (t.kind == RT_TEX_IMAGE) ARG_CHECK(t.image >= 0 && uint32_t(t.image) < d->n_images, "image index out of range");
    }
    std::vector<uint32_t> depth;
    rt_status st = checker_depths(d->textures, d->n_textures, depth);
    for (uint32_t i = 0; i < d->n_materials && st == RT_OK; ++i) st = check_material(d->materials[i], d->n_textures);
    for (uint32_t i = 0; i < d->n_spheres && st == RT_OK; ++i) st = check_sphere(d->spheres[i], d->n_materials);
    if (st != RT_OK) return st;
    ARG_CHECK(camera_finite(d->camera), "camera parameter is not finite");
    // resolve_texture (rt_shade.cuh) follows RT_MAX_CHECKER_DEPTH levels; the reference renders deeper chains, so they are
    // declined rather than rendered wrong (as trees deeper than RT_BVH_STACK_DEPTH are)
    for (uint32_t i = 0; i < d->n_textures; ++i)
        if (depth[i] > RT_MAX_CHECKER_DEPTH) {
            set_error("texture %u nests %u checker levels, more than RT_MAX_CHECKER_DEPTH (%d)", i, depth[i], RT_MAX_CHECKER_DEPTH);
            return RT_ERR_UNSUPPORTED;
        }
    return RT_OK;
}

// the device records (sph_a, sph_b, sph_c) of `count` spheres: record k is sphere spheres[src ? src[k] : k], whose list
// ordinal is ordinal[k].  k_apply packs the records of rt_scene_update_device on the device: the two packers must agree
// bit for bit (a scene's hits may not depend on which entry wrote its records).
void pack_spheres(const rt_sphere* spheres, const uint32_t* src, const uint32_t* ordinal, size_t count, float4* a, float4* b,
                  uint4* c) {
    {
        // c1 - c0 rounded toward zero (== __fsub_rz, vec3 operator- of moving_sphere::center, sphere.h:51).  The rounding
        // mode is switched once around this loop, not per operation: at 10^6 spheres a per-call switch
        // cost 150 ms of every scene upload.
        const int old_round = std::fegetround();
        std::fesetround(FE_TOWARDZERO);
        for (size_t k = 0; k < count; ++k) {
            const rt_sphere& sp = spheres[src ? src[k] : k];
            volatile float dx = sp.center1[0], dy = sp.center1[1], dz = sp.center1[2];
            dx = dx - sp.center0[0];
            dy = dy - sp.center0[1];
            dz = dz - sp.center0[2];
            b[k] = make_float4(dx, dy, dz, sp.time0);
        }
        std::fesetround(old_round);
    }
    for (size_t k = 0; k < count; ++k) {
        const rt_sphere& sp = spheres[src ? src[k] : k];
        a[k] = make_float4(sp.center0[0], sp.center0[1], sp.center0[2], sp.radius);
        float dt = sp.time1 - sp.time0; // FADD(RN) in the reference's SASS (sphere.h:51)
        uint32_t dt_bits;
        memcpy(&dt_bits, &dt, 4);
        c[k] = make_uint4(dt_bits, sp.material, sp.id, ordinal[k]);
    }
}

DMaterial pack_material(const rt_material& m) {
    return DMaterial{m.kind, m.texture, m.albedo[0], m.albedo[1], m.albedo[2], m.param, 0.f, 0.f};
}

// ---- rt_scene_update_device: the edit's records are read from device memory, checked, packed and scattered there ----

// one 48-byte rt_sphere as three 16-byte loads (the entry requires 16-byte aligned records)
__device__ __forceinline__ rt_sphere load_sphere(const rt_sphere* __restrict__ spheres, uint32_t j) {
    const float4* p = reinterpret_cast<const float4*>(spheres) + 3 * size_t(j);
    const float4 r0 = p[0], r1 = p[1], r2 = p[2];
    rt_sphere sp;
    sp.center0[0] = r0.x, sp.center0[1] = r0.y, sp.center0[2] = r0.z, sp.radius = r0.w;
    sp.center1[0] = r1.x, sp.center1[1] = r1.y, sp.center1[2] = r1.z, sp.time0 = r1.w;
    sp.time1 = r2.x, sp.material = __float_as_uint(r2.y), sp.id = __float_as_uint(r2.z), sp.flags = __float_as_uint(r2.w);
    return sp;
}

// where[list ordinal] = device index, from the ordinals the records carry
__global__ void __launch_bounds__(256) k_where(const uint4* __restrict__ sph_c, uint32_t n, uint32_t* __restrict__ where) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) where[sph_c[k].w] = k;
}

// claim[i] = the first edit position that names list ordinal i (claim starts at all ones)
__global__ void __launch_bounds__(256) k_claim(const uint32_t* __restrict__ idx, uint32_t m, uint32_t n, uint32_t* __restrict__ claim) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m && idx[j] < n) atomicMin(&claim[idx[j]], j);
}

// *verdict = min over the failing positions j of (j << 8 | rule): the lowest failing position and its first broken rule,
// whatever order the threads run in (starts at all ones)
__global__ void __launch_bounds__(256) k_check(const uint32_t* __restrict__ idx, const rt_sphere* __restrict__ spheres, uint32_t m,
                                               uint32_t n, uint32_t n_static, uint32_t n_materials, const uint32_t* __restrict__ claim,
                                               const uint32_t* __restrict__ where, unsigned long long* verdict) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t i = idx[j];
    const bool in = i < n;
    const uint32_t rule = sphere_edit_rule(load_sphere(spheres, j), i, n, in && claim[i] < j, in && where[i] >= n_static, n_materials);
    if (rule != SPH_OK) atomicMin(verdict, (static_cast<unsigned long long>(j) << 8) | rule);
}

// the checked records, packed as pack_spheres packs them, written at their device indices
__global__ void __launch_bounds__(256) k_apply(const uint32_t* __restrict__ idx, const rt_sphere* __restrict__ spheres, uint32_t m,
                                               const uint32_t* __restrict__ where, float4* __restrict__ a, float4* __restrict__ b,
                                               uint4* __restrict__ c) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t i = idx[j], k = where[i];
    const rt_sphere sp = load_sphere(spheres, j);
    a[k] = make_float4(sp.center0[0], sp.center0[1], sp.center0[2], sp.radius);
    b[k] = make_float4(__fsub_rz(sp.center1[0], sp.center0[0]), __fsub_rz(sp.center1[1], sp.center0[1]),
                       __fsub_rz(sp.center1[2], sp.center0[2]), sp.time0);
    c[k] = make_uint4(__float_as_uint(__fsub_rn(sp.time1, sp.time0)), sp.material, sp.id, i);
}

// ---- the emitter list, derived on the device at creation and after every update ----

// flag[list ordinal] = 1 when the sphere's material is an emitter
__global__ void __launch_bounds__(256) k_emitter_flags(const uint4* __restrict__ sph_c, uint32_t n, const DMaterial* __restrict__ mats,
                                                       uint32_t* __restrict__ flag) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint4 c = sph_c[k];
    flag[c.w] = mats[c.y].kind == RT_MAT_EMITTER ? 1u : 0u;
}

// lights[rank] = device index of the emitter of that rank in list order (pos: the exclusive sum of the flags), first
// RT_MAX_LIGHTS only
__global__ void __launch_bounds__(256) k_lights(const uint4* __restrict__ sph_c, uint32_t n, const DMaterial* __restrict__ mats,
                                                const uint32_t* __restrict__ pos, uint32_t* __restrict__ lights) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint4 c = sph_c[k];
    if (mats[c.y].kind == RT_MAT_EMITTER && pos[c.w] < RT_MAX_LIGHTS) lights[pos[c.w]] = k;
}

uint32_t blocks(uint32_t n) { return (n + 255) / 256; }

// the emitter spheres for RT_RENDER_EMITTER_SAMPLING (DScene::lights: device indices, the first RT_MAX_LIGHTS in list
// order) from the device records and materials; returns after one read-back of the list
rt_status find_lights(rt_scene* s, cudaStream_t st) {
    DScene& d = s->d;
    const uint32_t n = d.n_spheres;
    d.n_lights = 0;
    for (uint32_t k = 0; k < RT_MAX_LIGHTS; ++k) d.lights[k] = 0;
    if (n == 0) return RT_OK;
    PoolBuffer<uint32_t> buf; // flags, scan scratch, the list
    const size_t scratch = prims::scan_scratch_elems(n);
    CUDA_TRY(buf.alloc(n + scratch + RT_MAX_LIGHTS, st));
    uint32_t* flag = buf.get();
    uint32_t* lights = flag + n + scratch;
    CUDA_TRY(cudaMemsetAsync(lights, 0xFF, RT_MAX_LIGHTS * sizeof(uint32_t), st)); // unused entries: all ones
    k_emitter_flags<<<blocks(n), 256, 0, st>>>(d.sph_c, n, d.mats, flag);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(prims::exclusive_sum<uint32_t>(flag, flag, n, flag + n, st));
    k_lights<<<blocks(n), 256, 0, st>>>(d.sph_c, n, d.mats, flag, lights);
    CUDA_TRY(cudaGetLastError());
    uint32_t h[RT_MAX_LIGHTS];
    CUDA_TRY(cudaMemcpyAsync(h, lights, sizeof(h), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    while (d.n_lights < RT_MAX_LIGHTS && h[d.n_lights] != ~0u) {
        d.lights[d.n_lights] = h[d.n_lights];
        ++d.n_lights;
    }
    return RT_OK;
}

// the constant-bank copy of a brute-force list scene (DScene::lst_*) from the device records
rt_status read_list(rt_scene* s, cudaStream_t st) {
    DScene& d = s->d;
    if (d.n_list == 0) return RT_OK;
    float4 a[RT_LIST_MAX], b[RT_LIST_MAX];
    uint4 c[RT_LIST_MAX];
    CUDA_TRY(cudaMemcpyAsync(a, d.sph_a, d.n_list * sizeof(float4), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(b, d.sph_b, d.n_list * sizeof(float4), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(c, d.sph_c, d.n_list * sizeof(uint4), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (uint32_t k = 0; k < d.n_list; ++k) {
        d.lst_a[k] = a[k];
        d.lst_b[k] = b[k];
        memcpy(&d.lst_dt[k], &c[k].x, 4);
    }
    return RT_OK;
}

// the padded box of a sphere, over its whole motion when it moves
rth::Box sphere_box(const rt_sphere& sp) {
    return rth::sphere_box(sp.center0, (sp.flags & RT_SPHERE_MOVING) ? sp.center1 : sp.center0, sp.radius);
}

struct Tree {
    rth::BvhStats stats;              // depth of the deepest leaf, SAH cost
    float ms = 0.f;                   // the build's time: host clock (SAH), device events (LBVH)
    std::vector<rth::NodeHost> host;  // the SAH nodes, the source of an asynchronous copy
};

// The binary tree over the uploaded spheres (s->d.nodes, n_nodes, root): the host SAH build, or the LBVH with the chain of
// outsized spheres hung above its root.  order[k] is the description index of device record k.
rt_status build_tree(rt_scene* s, const rt_scene_desc* desc, uint32_t mode, const std::vector<uint32_t>& order, Tree& t) {
    DScene& d = s->d;
    const uint32_t n = d.n_spheres;
    const cudaStream_t stream = s->ctx->stream;
    BvhNode* nodes = nullptr;
    rt_status st;
    if (mode == RT_BVH_HOST_SAH) {
        std::vector<rth::Box> boxes(n);
        for (uint32_t k = 0; k < n; ++k) boxes[k] = sphere_box(desc->spheres[order[k]]);
        const auto t0 = std::chrono::steady_clock::now();
        rth::build_bvh_sah(boxes, t.host, &t.stats);
        t.ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if ((st = dev_alloc(s, &nodes, t.host.size())) != RT_OK) return st;
        d.nodes = nodes;
        d.n_nodes = uint32_t(t.host.size());
        CUDA_TRY(cudaMemcpyAsync(nodes, t.host.data(), t.host.size() * sizeof(BvhNode), cudaMemcpyHostToDevice, stream));
        return RT_OK;
    }
    if (mode != RT_BVH_GPU_LBVH) return RT_OK;
    if ((st = dev_alloc(s, &nodes, n - 1)) != RT_OK) return st;
    d.nodes = nodes;
    d.n_nodes = n - 1;
    // Outsized primitives (the r = 1000 ground every scene of this renderer has) would sit deep in a Morton-ordered
    // tree and inflate the boxes of all their ancestors, so every ray would walk that whole chain.  They are kept
    // out of the LBVH and hung above its root instead: root -> (big_k, (... (big_0, LBVH root))).
    std::vector<uint32_t> big, normal;
    {
        std::vector<float> radii(n);
        for (uint32_t k = 0; k < n; ++k) radii[k] = std::fabs(desc->spheres[order[k]].radius);
        std::vector<float> tmp(radii);
        std::nth_element(tmp.begin(), tmp.begin() + n / 2, tmp.end());
        const float limit = 32.f * tmp[n / 2];
        for (uint32_t k = 0; k < n; ++k) (radii[k] > limit && big.size() < 32 ? big : normal).push_back(k);
        if (normal.size() < 2) { // nothing sensible to separate
            big.clear();
            normal.clear();
        }
    }
    const uint32_t m = big.empty() ? n : uint32_t(normal.size());
    PoolBuffer<uint32_t> d_ids;
    if (!big.empty()) {
        CUDA_TRY(d_ids.alloc(m, stream));
        CUDA_TRY(cudaMemcpyAsync(d_ids.get(), normal.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
    }
    float rb[6];
    const cudaError_t e = lbvh_build(d.sph_a, d.sph_b, d.n_static, d_ids.get(), m, nodes, stream, &t.ms, &t.stats.depth, rb);
    if (e != cudaSuccess) {
        set_error("GPU LBVH build failed: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    if (big.empty()) return RT_OK;
    std::vector<rth::NodeHost> chain(big.size());
    rth::Box below{{rb[0], rb[1], rb[2]}, {rb[3], rb[4], rb[5]}};
    int32_t below_ref = 0; // the LBVH root
    for (size_t k = 0; k < big.size(); ++k) {
        const rth::Box bb = sphere_box(desc->spheres[order[big[k]]]);
        rth::NodeHost& nd = chain[k];
        for (int a = 0; a < 3; ++a) {
            nd.lmin[a] = bb.lo[a];
            nd.lmax[a] = bb.hi[a];
            nd.rmin[a] = below.lo[a];
            nd.rmax[a] = below.hi[a];
            below.lo[a] = std::min(below.lo[a], bb.lo[a]);
            below.hi[a] = std::max(below.hi[a], bb.hi[a]);
        }
        nd.left = ~int32_t(big[k]);
        nd.right = below_ref;
        nd.pad0 = nd.pad1 = 0.f;
        below_ref = int32_t(m - 1 + k);
    }
    CUDA_TRY(cudaMemcpyAsync(nodes + (m - 1), chain.data(), chain.size() * sizeof(BvhNode), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(cudaStreamSynchronize(stream)); // `chain` is a pageable host buffer
    d.root = uint32_t(below_ref);
    t.stats.depth += uint32_t(big.size());
    return RT_OK;
}

// The forms the walks read, from the finished binary nodes (s->d.nodes, n_nodes, root; depth: the build's): the centre /
// half-extent nodes, the 4-wide nodes and their 64-byte quantised form.  The first call (scene creation) allocates them;
// later calls (after a refit) overwrite them in place.
rt_status derive_forms(rt_scene* s, uint32_t depth, cudaStream_t st) {
    DScene& d = s->d;
    const bool first = d.nodes_ch == nullptr;
    const uint32_t n_nodes = d.n_nodes, room4 = n_nodes / 2 + 64;
    rt_status rs;
    if (first && (rs = dev_alloc(s, &d.nodes_ch, n_nodes)) != RT_OK) return rs;
    cudaError_t e = bvh_nodes_ch(d.nodes, n_nodes, const_cast<BvhNodeCH*>(d.nodes_ch), st);
    if (e != cudaSuccess) {
        set_error("BVH node conversion failed: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    // the 4-wide form the persistent-lane kernel walks (half the dependent node fetches per ray)
    if (first && (rs = dev_alloc(s, &d.nodes4, room4)) != RT_OK) return rs;
    PoolBuffer<BvhNode4> scratch; // worst case (a degenerate chain) every binary node survives
    CUDA_TRY(scratch.alloc(n_nodes, st));
    uint32_t n4 = 0, root4 = 0;
    e = bvh_collapse4(d.nodes, n_nodes, d.root, depth, scratch.get(), &n4, &root4, st);
    if (e == cudaSuccess && !first && (n4 != d.n_nodes4 || root4 != d.root4)) { // a refit keeps the topology and its numbering
        set_error("4-wide BVH collapse gave %u nodes (root %u), the scene has %u (root %u)", n4, root4, d.n_nodes4, d.root4);
        return RT_ERR_CUDA;
    }
    if (e == cudaSuccess && first && n4 > room4) { // unusually deep tree: keep the big array itself
        s->allocs.push_back(scratch.get());
        d.nodes4 = scratch.release();
    } else if (e == cudaSuccess) {
        e = cudaMemcpyAsync(const_cast<BvhNode4*>(d.nodes4), scratch.get(), size_t(n4) * sizeof(BvhNode4), cudaMemcpyDeviceToDevice, st);
    }
    if (e != cudaSuccess) {
        set_error("4-wide BVH collapse failed: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    d.n_nodes4 = n4;
    d.root4 = root4;
    // ... and its 64-byte quantised form, walked only when it represents every node (the memory stays with the scene)
    d.nodes4q = nullptr;
    if (n4 && !getenv("RT_NO_BVH4Q") && (first || s->nodes4q_mem)) {
        if (first && (rs = dev_alloc(s, &s->nodes4q_mem, n4)) != RT_OK) return rs;
        bool quant_ok = false;
        e = bvh_quantize4(d.nodes4, n4, s->nodes4q_mem, &quant_ok, st);
        if (e != cudaSuccess) {
            set_error("4-wide BVH quantisation failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
        if (quant_ok) d.nodes4q = s->nodes4q_mem;
    }
    return RT_OK;
}

rt_status upload_materials(rt_scene* s, const rt_scene_desc* desc, cudaStream_t stream) {
    std::vector<DMaterial> hm(desc->n_materials);
    for (uint32_t i = 0; i < desc->n_materials; ++i) hm[i] = pack_material(desc->materials[i]);
    std::vector<DTexture> ht(desc->n_textures);
    for (uint32_t i = 0; i < desc->n_textures; ++i) {
        const rt_texture& t = desc->textures[i];
        ht[i] = DTexture{t.kind,      t.even,      t.odd,       t.image,   t.color1[0], t.color1[1],
                         t.color1[2], t.density,   t.color2[0], t.color2[1], t.color2[2], t.hardness};
    }
    DMaterial* dmats = nullptr;
    DTexture* dtexs = nullptr;
    rt_status st;
    if ((st = dev_alloc(s, &dmats, hm.size())) != RT_OK) return st;
    if ((st = dev_alloc(s, &dtexs, ht.size())) != RT_OK) return st;
    if (!hm.empty()) CUDA_TRY(cudaMemcpyAsync(dmats, hm.data(), hm.size() * sizeof(DMaterial), cudaMemcpyHostToDevice, stream));
    if (!ht.empty()) CUDA_TRY(cudaMemcpyAsync(dtexs, ht.data(), ht.size() * sizeof(DTexture), cudaMemcpyHostToDevice, stream));
    s->d.mats = dmats;
    s->d.texs = dtexs;
    return RT_OK;
}

// image textures: float RGB -> float4 cudaArray (from the context's cache of destroyed scenes' arrays when one has the
// size) + point-sampled texture object
rt_status upload_images(rt_scene* s, const rt_scene_desc* desc, cudaStream_t stream) {
    rt_context* ctx = s->ctx;
    for (uint32_t i = 0; i < desc->n_images; ++i) {
        const rt_image& im = desc->images[i];
        const size_t texels = size_t(im.width) * size_t(im.height);
        PoolBuffer<float> d_rgb;
        PoolBuffer<float4> d_rgba;
        CUDA_TRY(d_rgb.alloc(texels * 3, stream));
        cudaError_t e = d_rgba.alloc(texels, stream);
        if (e != cudaSuccess) {
            set_error("cudaMallocAsync(image staging) failed: %s", cudaGetErrorString(e));
            return RT_ERR_OOM;
        }
        cudaArray_t arr = nullptr;
        {
            std::lock_guard<std::mutex> lock(ctx->cache_mutex);
            for (size_t k = 0; k < ctx->array_cache.size(); ++k)
                if (ctx->array_cache[k].width == im.width && ctx->array_cache[k].height == im.height) {
                    arr = ctx->array_cache[k].arr;
                    ctx->array_cache.erase(ctx->array_cache.begin() + long(k));
                    break;
                }
        }
        cudaChannelFormatDesc cd = cudaCreateChannelDesc<float4>();
        e = cudaMemcpyAsync(d_rgb.get(), im.rgb, texels * 3 * sizeof(float), cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) {
            launch_rgb_to_rgba(d_rgb.get(), d_rgba.get(), texels, ctx->sm_count, stream);
            if (!arr) e = cudaMallocArray(&arr, &cd, size_t(im.width), size_t(im.height));
        }
        if (e == cudaSuccess) {
            s->arrays.push_back(rt_context::CachedArray{im.width, im.height, arr});
            e = cudaMemcpy2DToArrayAsync(arr, 0, 0, d_rgba.get(), size_t(im.width) * sizeof(float4), size_t(im.width) * sizeof(float4),
                                         size_t(im.height), cudaMemcpyDeviceToDevice, stream);
        }
        if (e != cudaSuccess) {
            set_error("image texture upload failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
        cudaResourceDesc rd{};
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        cudaTextureDesc td{};
        td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp;
        td.filterMode = cudaFilterModePoint;
        td.readMode = cudaReadModeElementType;
        td.normalizedCoords = 0;
        cudaTextureObject_t tex = 0;
        CUDA_TRY(cudaCreateTextureObject(&tex, &rd, &td, nullptr));
        s->texobjs.push_back(tex);
        s->d.images[i] = DImage{tex, im.width, im.height};
        s->info.device_bytes += texels * sizeof(float4);
    }
    return RT_OK;
}

// Every argument of an edit, before any device work (so a refused edit leaves the scene as it was).
rt_status check_edit(const rt_context* ctx, const rt_scene* s, const rt_scene_edit* e) {
    ARG_CHECK(ctx && s && e, "ctx/scene/edit is NULL");
    ARG_CHECK(s->ctx == ctx, "the scene belongs to another context");
    ARG_CHECK(e->n_spheres == 0 || (e->sphere_index && e->spheres), "sphere_index/spheres is NULL");
    ARG_CHECK(e->n_materials == 0 || (e->material_index && e->materials), "material_index/materials is NULL");
    const uint32_t n = s->d.n_spheres, n_mat = s->n_materials;
    std::vector<bool> seen(e->n_spheres ? n : 0);
    for (uint32_t j = 0; j < e->n_spheres; ++j) {
        const uint32_t i = e->sphere_index[j];
        const bool in = i < n;
        const uint32_t r = sphere_edit_rule(e->spheres[j], i, n, in && seen[i], in && s->where[i] >= s->d.n_static, n_mat);
        ARG_CHECK(r == SPH_OK, kSphereRuleMessage[r]);
        seen[i] = true;
    }
    seen.assign(e->n_materials ? n_mat : 0, false);
    for (uint32_t j = 0; j < e->n_materials; ++j) {
        const uint32_t i = e->material_index[j];
        ARG_CHECK(i < n_mat, "material index out of range");
        ARG_CHECK(!seen[i], "material index repeated");
        seen[i] = true;
        const rt_status st = check_material(e->materials[j], s->n_textures);
        if (st != RT_OK) return st;
    }
    ARG_CHECK(!e->camera || camera_finite(*e->camera), "camera parameter is not finite");
    return RT_OK;
}

// Sphere and material records: packed on the host, one copy of the records and one of their device indices, a scatter.
rt_status upload_records(rt_scene* s, const rt_scene_edit* e, cudaStream_t st) {
    const uint32_t m = e->n_spheres, k = e->n_materials;
    std::vector<float4> rec(size_t(m) * 3); // sph_a records, sph_b records, sph_c records
    std::vector<uint32_t> idx(size_t(m) + k); // their device indices, then the material indices
    std::vector<DMaterial> mats(k);
    float4* a = rec.data();
    float4* b = a + m;
    uint4* c = reinterpret_cast<uint4*>(b + m);
    pack_spheres(e->spheres, nullptr, e->sphere_index, m, a, b, c);
    for (uint32_t j = 0; j < m; ++j) idx[j] = s->where[e->sphere_index[j]];
    for (uint32_t j = 0; j < k; ++j) {
        mats[j] = pack_material(e->materials[j]);
        idx[m + j] = e->material_index[j];
    }
    PoolBuffer<float4> d_rec;
    PoolBuffer<DMaterial> d_mats;
    PoolBuffer<uint32_t> d_idx;
    CUDA_TRY(d_idx.alloc(idx.size(), st));
    CUDA_TRY(cudaMemcpyAsync(d_idx.get(), idx.data(), idx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    if (m) {
        CUDA_TRY(d_rec.alloc(rec.size(), st));
        CUDA_TRY(cudaMemcpyAsync(d_rec.get(), rec.data(), rec.size() * sizeof(float4), cudaMemcpyHostToDevice, st));
        const float4* da = d_rec.get();
        launch_scatter(da, d_idx.get(), m, const_cast<float4*>(s->d.sph_a), st);
        launch_scatter(da + m, d_idx.get(), m, const_cast<float4*>(s->d.sph_b), st);
        launch_scatter(reinterpret_cast<const uint4*>(da + 2 * size_t(m)), d_idx.get(), m, const_cast<uint4*>(s->d.sph_c), st);
    }
    if (k) {
        CUDA_TRY(d_mats.alloc(k, st));
        CUDA_TRY(cudaMemcpyAsync(d_mats.get(), mats.data(), k * sizeof(DMaterial), cudaMemcpyHostToDevice, st));
        launch_scatter<DMaterial>(d_mats.get(), d_idx.get() + m, k, const_cast<DMaterial*>(s->d.mats), st);
    }
    CUDA_TRY(cudaGetLastError());
    // the host copy of the records goes out of scope: the copies from it must have been made
    CUDA_TRY(cudaStreamSynchronize(st));
    return RT_OK;
}

// The sphere records of rt_scene_update_device, from device memory: checked on the device (the verdict comes back in one
// copy; nothing of the scene is written before it), then packed and scattered.
rt_status apply_device_records(rt_scene* s, const uint32_t* idx, const rt_sphere* spheres, uint32_t m, cudaStream_t st) {
    DScene& d = s->d;
    const uint32_t n = d.n_spheres;
    ARG_CHECK(n != 0, kSphereRuleMessage[SPH_INDEX_RANGE]); // (every index of an edit of an empty scene is out of range)
    if (!s->where_dev) { // first device update of this scene: list ordinal -> device index, kept with the scene
        void* p = nullptr;
        CUDA_TRY(cudaMallocFromPoolAsync(&p, size_t(n) * sizeof(uint32_t), s->ctx->pool, st));
        s->allocs.push_back(p);
        s->where_dev = static_cast<uint32_t*>(p);
        k_where<<<blocks(n), 256, 0, st>>>(d.sph_c, n, s->where_dev);
        CUDA_TRY(cudaGetLastError());
    }
    PoolBuffer<unsigned long long> verdict;
    PoolBuffer<uint32_t> claim;
    CUDA_TRY(verdict.alloc(1, st));
    CUDA_TRY(claim.alloc(n, st));
    CUDA_TRY(cudaMemsetAsync(verdict.get(), 0xFF, sizeof(unsigned long long), st));
    CUDA_TRY(cudaMemsetAsync(claim.get(), 0xFF, size_t(n) * sizeof(uint32_t), st));
    k_claim<<<blocks(m), 256, 0, st>>>(idx, m, n, claim.get());
    k_check<<<blocks(m), 256, 0, st>>>(idx, spheres, m, n, d.n_static, s->n_materials, claim.get(), s->where_dev, verdict.get());
    CUDA_TRY(cudaGetLastError());
    unsigned long long v = 0;
    CUDA_TRY(cudaMemcpyAsync(&v, verdict.get(), sizeof(v), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    ARG_CHECK(v == ~0ull, kSphereRuleMessage[v & 0xFF]);
    k_apply<<<blocks(m), 256, 0, st>>>(idx, spheres, m, s->where_dev, const_cast<float4*>(d.sph_a), const_cast<float4*>(d.sph_b),
                                       const_cast<uint4*>(d.sph_c));
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

// The binary node boxes from the current primitives, bottom-up over the whole tree, then every form derived from them.
rt_status refit(rt_scene* s, cudaStream_t st) {
    DScene& d = s->d;
    BvhNode* nodes = const_cast<BvhNode*>(d.nodes);
    if (!s->parents) { // first refit of this scene: the parent table, kept with the scene (not counted in info.device_bytes)
        void* p = nullptr;
        CUDA_TRY(cudaMallocFromPoolAsync(&p, (size_t(d.n_nodes) + d.n_spheres) * sizeof(int), s->ctx->pool, st));
        s->allocs.push_back(p);
        uint32_t levels = 0;
        CUDA_TRY(bvh_parents(nodes, d.n_nodes, d.n_spheres, static_cast<int*>(p), &levels, st));
        if (levels != s->info.bvh_depth) {
            set_error("scene update: the parent table has %u levels, the tree was built with %u", levels, s->info.bvh_depth);
            return RT_ERR_CUDA;
        }
        s->parents = static_cast<int*>(p);
    }
    CUDA_TRY(bvh_refit(d.sph_a, d.sph_b, d.n_spheres, d.n_static, nodes, d.n_nodes, s->parents, st));
    return derive_forms(s, s->info.bvh_depth, st);
}

// The update both entries share: `write_records(stream)` enqueues the writes of the edit's records (or refuses the edit
// before it writes anything), then the refit when spheres changed, inside the window ms_device times; then the host state
// that depends on the records: the constant-bank list and the emitter list.  Returns when the update is complete.
template <class WriteRecords>
rt_status apply_update(rt_scene* s, bool spheres, WriteRecords&& write_records, float* ms_device) {
    const cudaStream_t st = s->ctx->stream;
    TimingEvent e0, e1;
    CUDA_TRY(e0.create());
    CUDA_TRY(e1.create());
    CUDA_TRY(cudaEventRecord(e0.ev, st));
    rt_status rs = write_records(st);
    if (rs != RT_OK) return rs;
    if (spheres && s->d.nodes && (rs = refit(s, st)) != RT_OK) return rs;
    CUDA_TRY(cudaEventRecord(e1.ev, st));
    CUDA_TRY(cudaEventSynchronize(e1.ev)); // (the reads below may enqueue nothing: a scene without spheres)
    if (spheres && (rs = read_list(s, st)) != RT_OK) return rs;
    if ((rs = find_lights(s, st)) != RT_OK) return rs;
    if (ms_device) CUDA_TRY(cudaEventElapsedTime(ms_device, e0.ev, e1.ev));
    return RT_OK;
}

} // namespace

// every parameter of a camera finite (scene descriptions, frame sequences, rt_orbit_cameras)
bool camera_finite(const rt_camera& c) {
    return finite3(c.lookfrom) && finite3(c.lookat) && finite3(c.up) && finite1(c.vfov) && finite1(c.aspect) && finite1(c.aperture) &&
           finite1(c.focus_dist) && finite1(c.time0) && finite1(c.time1);
}

} // namespace rtd

using namespace rtd;

extern "C" rt_status rt_scene_create(rt_context* ctx, const rt_scene_desc* desc, rt_scene** out) try {
    ARG_CHECK(ctx != nullptr && out != nullptr, "ctx/out is NULL");
    *out = nullptr;
    rt_status st = validate_desc(desc);
    if (st != RT_OK) return st;
    st = make_current(ctx);
    if (st != RT_OK) return st;

    rt_scene* s = new (std::nothrow) rt_scene();
    if (!s) return RT_ERR_OOM;
    s->ctx = ctx;
    struct Guard {
        rt_scene* s;
        ~Guard() {
            if (s) rt_scene_destroy(s);
        }
    } guard{s};

    const auto t_begin = std::chrono::steady_clock::now();
    const uint32_t n = desc->n_spheres;
    const cudaStream_t stream = ctx->stream;
    uint32_t mode = desc->bvh_mode;
    if (mode == RT_BVH_AUTO) mode = n <= 12 ? RT_BVH_NONE : (n <= 200000 ? RT_BVH_HOST_SAH : RT_BVH_GPU_LBVH);
    if (n < 2) mode = RT_BVH_NONE;

    // ---- order and pack: static spheres first (stable), SoA float4 records ----
    std::vector<uint32_t> order;
    order.reserve(n);
    for (uint32_t i = 0; i < n; ++i)
        if (!(desc->spheres[i].flags & RT_SPHERE_MOVING)) order.push_back(i);
    const uint32_t n_static = uint32_t(order.size());
    for (uint32_t i = 0; i < n; ++i)
        if (desc->spheres[i].flags & RT_SPHERE_MOVING) order.push_back(i);
    std::vector<float4> ha(n), hb(n);
    std::vector<uint4> hc(n);
    pack_spheres(desc->spheres, order.data(), order.data(), n, ha.data(), hb.data(), hc.data());
    float4 *da = nullptr, *db = nullptr;
    uint4* dc = nullptr;
    if ((st = dev_alloc(s, &da, n)) != RT_OK) return st;
    if ((st = dev_alloc(s, &db, n)) != RT_OK) return st;
    if ((st = dev_alloc(s, &dc, n)) != RT_OK) return st;
    if (n) {
        CUDA_TRY(cudaMemcpyAsync(da, ha.data(), n * sizeof(float4), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(db, hb.data(), n * sizeof(float4), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dc, hc.data(), n * sizeof(uint4), cudaMemcpyHostToDevice, stream));
    }
    s->d.sph_a = da;
    s->d.sph_b = db;
    s->d.sph_c = dc;
    s->d.n_spheres = n;
    s->d.n_static = n_static;

    // ---- the tree, refused before anything is derived from it when a walk's stack cannot hold it ----
    Tree tree;
    if ((st = build_tree(s, desc, mode, order, tree)) != RT_OK) return st;
    if (tree.stats.depth > RT_BVH_STACK_DEPTH) {
        set_error("BVH depth %u exceeds the traversal stack (%d)", tree.stats.depth, RT_BVH_STACK_DEPTH);
        return RT_ERR_UNSUPPORTED;
    }
    if (s->d.nodes && (st = derive_forms(s, tree.stats.depth, stream)) != RT_OK) return st;
    if ((st = upload_materials(s, desc, stream)) != RT_OK) return st;
    if ((st = upload_images(s, desc, stream)) != RT_OK) return st;

    // ---- what the kernels read besides the device arrays, the mirrors rt_scene_update needs, and the scene's info ----
    // the list in the constant bank (DScene::lst_*) and the emitter list come from the device records, as after an update
    s->d.n_list = mode == RT_BVH_NONE && n <= RT_LIST_MAX ? n : 0;
    if ((st = read_list(s, stream)) != RT_OK) return st;
    if ((st = find_lights(s, stream)) != RT_OK) return st;
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());
    s->d.has_noise = 0;
    for (uint32_t i = 0; i < desc->n_textures; ++i) {
        const uint32_t kind = desc->textures[i].kind;
        if (kind == RT_TEX_NOISE_PERLIN || kind == RT_TEX_NOISE_TURBULANCE || kind == RT_TEX_NOISE_MARBLE || kind == RT_TEX_WOOD) s->d.has_noise = 1;
    }
    make_camera(desc->camera, s->d.cam);
    s->where.resize(n); // list ordinal -> device index
    for (uint32_t k = 0; k < n; ++k) s->where[order[k]] = k;
    s->n_materials = desc->n_materials;
    s->n_textures = desc->n_textures;

    const auto t_end = std::chrono::steady_clock::now();
    s->info.n_spheres = n;
    s->info.n_nodes = s->d.n_nodes;
    s->info.bvh_mode = mode;
    s->info.bvh_depth = tree.stats.depth;
    s->info.sah_cost = tree.stats.sah_cost;
    s->info.ms_build = tree.ms;
    s->info.ms_upload = std::chrono::duration<float, std::milli>(t_end - t_begin).count() - (mode == RT_BVH_HOST_SAH ? tree.ms : 0.f);
    guard.s = nullptr;
    *out = s;
    return RT_OK;
}
RT_API_CATCH

extern "C" void rt_scene_destroy(rt_scene* scene) {
    if (!scene) return;
    if (scene->ctx) cudaSetDevice(scene->ctx->device);
    // the scene's kernels are ordered before these on the context stream
    for (auto t : scene->texobjs) cudaDestroyTextureObject(t);
    for (auto& a : scene->arrays) {
        bool kept = false;
        if (scene->ctx) {
            std::lock_guard<std::mutex> lock(scene->ctx->cache_mutex);
            if (scene->ctx->array_cache.size() < 8) {
                scene->ctx->array_cache.push_back(a);
                kept = true;
            }
        }
        if (!kept) cudaFreeArray(a.arr);
    }
    for (auto p : scene->allocs) {
        if (scene->ctx) cudaFreeAsync(p, scene->ctx->stream);
        else cudaFree(p);
    }
    delete scene;
}

extern "C" rt_status rt_scene_get_info(const rt_scene* scene, rt_scene_info* info) try {
    ARG_CHECK(scene && info, "scene/info is NULL");
    *info = scene->info;
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_scene_update(rt_context* ctx, rt_scene* scene, const rt_scene_edit* edit, float* ms_device) try {
    if (ms_device) *ms_device = 0.f;
    rt_status st = check_edit(ctx, scene, edit);
    if (st != RT_OK) return st;
    if (edit->camera) make_camera(*edit->camera, scene->d.cam);
    if (edit->n_spheres == 0 && edit->n_materials == 0) return RT_OK;
    if ((st = make_current(ctx)) != RT_OK) return st;
    return apply_update(scene, edit->n_spheres != 0, [&](cudaStream_t s) { return upload_records(scene, edit, s); }, ms_device);
}
RT_API_CATCH

extern "C" rt_status rt_scene_update_device(rt_context* ctx, rt_scene* scene, const uint32_t* sphere_index_dev,
                                            const rt_sphere* spheres_dev, uint32_t n_spheres, float* ms_device) try {
    if (ms_device) *ms_device = 0.f;
    ARG_CHECK(ctx && scene, "ctx/scene is NULL");
    ARG_CHECK(n_spheres == 0 || (sphere_index_dev && spheres_dev), "sphere_index_dev/spheres_dev is NULL");
    ARG_CHECK(scene->ctx == ctx, "the scene belongs to another context");
    if (n_spheres == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    // a pointer no kernel of ctx's device may read is refused here, never handed to a kernel
    for (const void* p : {static_cast<const void*>(sphere_index_dev), static_cast<const void*>(spheres_dev)}) {
        cudaPointerAttributes at{};
        const cudaError_t e = cudaPointerGetAttributes(&at, p);
        if (e != cudaSuccess) cudaGetLastError(); // (clears the error: the call only asked)
        ARG_CHECK(e == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == ctx->device,
                  "sphere_index_dev/spheres_dev is not device or managed memory of the context's device");
    }
    ARG_CHECK(reinterpret_cast<uintptr_t>(spheres_dev) % 16 == 0, "spheres_dev is not 16-byte aligned");
    ARG_CHECK(reinterpret_cast<uintptr_t>(sphere_index_dev) % 4 == 0, "sphere_index_dev is not 4-byte aligned");
    return apply_update(
        scene, true, [&](cudaStream_t s) { return apply_device_records(scene, sphere_index_dev, spheres_dev, n_spheres, s); }, ms_device);
}
RT_API_CATCH
