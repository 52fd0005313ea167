// rt_update.cu — rt_scene_update: edits of a resident scene (sphere records, material records, the camera) and the refit of
// every node form of its tree on the device.  The tree's topology stays as it was built; only its boxes change
// (DESIGN.md "Scene updates").
#include <cstdlib>
#include <cstring>
#include <vector>

#include "rt_internal.hpp"
#include "rt_lbvh.cuh"

namespace rtd {
namespace {

// dst[idx[j]] = src[j]
template <class T>
__global__ void __launch_bounds__(256) k_scatter(const T* __restrict__ src, const uint32_t* __restrict__ idx, uint32_t n, T* __restrict__ dst) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) dst[idx[j]] = src[j];
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

// the number of levels: the most inner nodes on a path from a primitive to the root
__global__ void __launch_bounds__(256) k_levels(uint32_t n, const int* __restrict__ parent_inner, const int* __restrict__ parent_leaf,
                                                unsigned* __restrict__ levels) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned d = 0;
    if (k < n)
        for (int p = parent_leaf[k]; p >= 0; p = parent_inner[p]) ++d;
    d = __reduce_max_sync(0xffffffffu, d);
    if ((threadIdx.x & 31) == 0) atomicMax(levels, d);
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

template <class T>
void launch_scatter(const T* src, const uint32_t* idx, uint32_t n, T* dst, cudaStream_t st) {
    if (n) k_scatter<T><<<(n + 255) / 256, 256, 0, st>>>(src, idx, n, dst);
}

// Every argument of an edit, before any device work (so a refused edit leaves the scene as it was).
rt_status check_edit(const rt_context* ctx, const rt_scene* s, const rt_scene_edit* e) {
    ARG_CHECK(ctx && s && e, "ctx/scene/edit is NULL");
    ARG_CHECK(s->ctx == ctx, "the scene belongs to another context");
    ARG_CHECK(e->n_spheres == 0 || (e->sphere_index && e->spheres), "sphere_index/spheres is NULL");
    ARG_CHECK(e->n_materials == 0 || (e->material_index && e->materials), "material_index/materials is NULL");
    const uint32_t n = s->d.n_spheres, n_mat = uint32_t(s->material_kind.size());
    std::vector<bool> seen(e->n_spheres ? n : 0);
    for (uint32_t j = 0; j < e->n_spheres; ++j) {
        const uint32_t i = e->sphere_index[j];
        ARG_CHECK(i < n, "sphere index out of range");
        ARG_CHECK(!seen[i], "sphere index repeated");
        seen[i] = true;
        // static spheres are stored before the moving ones: a sphere keeps its kind
        ARG_CHECK(((e->spheres[j].flags & RT_SPHERE_MOVING) != 0) == (s->where[i] >= s->d.n_static),
                  "an edit cannot make a static sphere moving or a moving one static");
        const rt_status st = check_sphere(e->spheres[j], n_mat);
        if (st != RT_OK) return st;
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
    // the brute-force list's copy in the kernel parameters
    for (uint32_t j = 0; j < m && s->d.n_list; ++j) {
        const uint32_t i = idx[j];
        s->d.lst_a[i] = a[j];
        s->d.lst_b[i] = b[j];
        memcpy(&s->d.lst_dt[i], &c[j].x, 4);
    }
    // the host copy of the records goes out of scope: the copies from it must have been made
    CUDA_TRY(cudaStreamSynchronize(st));
    return RT_OK;
}

// The binary node boxes from the current primitives, bottom-up over the whole tree, then every form derived from them.
rt_status refit(rt_scene* s, cudaStream_t st) {
    DScene& d = s->d;
    const uint32_t n = d.n_spheres, n_nodes = d.n_nodes;
    BvhNode* nodes = const_cast<BvhNode*>(d.nodes);
    if (!s->parents) { // first refit of this scene: the parent table, kept with the scene
        void* p = nullptr;
        CUDA_TRY(cudaMallocFromPoolAsync(&p, (size_t(n_nodes) + n) * sizeof(int), s->ctx->pool, st));
        s->allocs.push_back(p);
        int* parents = static_cast<int*>(p);
        PoolBuffer<unsigned> d_levels;
        CUDA_TRY(d_levels.alloc(1, st));
        CUDA_TRY(cudaMemsetAsync(parents, 0xff, (size_t(n_nodes) + n) * sizeof(int), st));
        CUDA_TRY(cudaMemsetAsync(d_levels.get(), 0, sizeof(unsigned), st));
        k_parents<<<(n_nodes + 255) / 256, 256, 0, st>>>(nodes, n_nodes, parents, parents + n_nodes);
        k_levels<<<(n + 255) / 256, 256, 0, st>>>(n, parents, parents + n_nodes, d_levels.get());
        CUDA_TRY(cudaGetLastError());
        unsigned levels = 0;
        CUDA_TRY(cudaMemcpyAsync(&levels, d_levels.get(), sizeof levels, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (levels != s->info.bvh_depth) {
            set_error("scene update: the parent table has %u levels, the tree was built with %u", levels, s->info.bvh_depth);
            return RT_ERR_CUDA;
        }
        s->parents = parents;
    }
    PoolBuffer<unsigned> visits;
    CUDA_TRY(visits.alloc(n_nodes, st));
    CUDA_TRY(cudaMemsetAsync(visits.get(), 0, n_nodes * sizeof(unsigned), st));
    k_refit_all<<<(n + 255) / 256, 256, 0, st>>>(d.sph_a, d.sph_b, n, d.n_static, nodes, s->parents, s->parents + n_nodes, visits.get());
    CUDA_TRY(cudaGetLastError());

    cudaError_t e = bvh_nodes_ch(nodes, n_nodes, const_cast<BvhNodeCH*>(d.nodes_ch), st);
    if (e != cudaSuccess) {
        set_error("scene update: BVH node conversion failed: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    PoolBuffer<BvhNode4> scratch;
    CUDA_TRY(scratch.alloc(n_nodes, st));
    uint32_t n4 = 0, root4 = 0;
    e = bvh_collapse4(nodes, n_nodes, d.root, s->info.bvh_depth, scratch.get(), &n4, &root4, st);
    if (e != cudaSuccess) {
        set_error("scene update: 4-wide BVH collapse failed: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    if (n4 != d.n_nodes4 || root4 != d.root4) { // the topology is unchanged, so is the 4-wide numbering
        set_error("scene update: the 4-wide collapse gave %u nodes (root %u), the scene has %u (root %u)", n4, root4, d.n_nodes4, d.root4);
        return RT_ERR_CUDA;
    }
    CUDA_TRY(cudaMemcpyAsync(const_cast<BvhNode4*>(d.nodes4), scratch.get(), size_t(n4) * sizeof(BvhNode4), cudaMemcpyDeviceToDevice, st));
    d.nodes4q = nullptr; // until the quantised nodes are known to hold the new boxes
    if (s->nodes4q_mem && !getenv("RT_NO_BVH4Q")) {
        bool quant_ok = false;
        e = bvh_quantize4(d.nodes4, n4, s->nodes4q_mem, &quant_ok, st);
        if (e != cudaSuccess) {
            set_error("scene update: 4-wide BVH quantisation failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
        if (quant_ok) d.nodes4q = s->nodes4q_mem;
    }
    return RT_OK;
}

} // namespace
} // namespace rtd

extern "C" rt_status rt_scene_update(rt_context* ctx, rt_scene* scene, const rt_scene_edit* edit, float* ms_device) try {
    if (ms_device) *ms_device = 0.f;
    rt_status st = rtd::check_edit(ctx, scene, edit);
    if (st != RT_OK) return st;
    if (edit->camera) rtd::make_camera(*edit->camera, scene->d.cam);
    if (edit->n_spheres == 0 && edit->n_materials == 0) return RT_OK;
    if ((st = rtd::make_current(ctx)) != RT_OK) return st;
    const cudaStream_t stream = ctx->stream;
    rtd::TimingEvent e0, e1;
    CUDA_TRY(e0.create());
    CUDA_TRY(e1.create());
    CUDA_TRY(cudaEventRecord(e0.ev, stream));
    if ((st = rtd::upload_records(scene, edit, stream)) != RT_OK) return st;
    if (edit->n_spheres && scene->d.nodes && (st = rtd::refit(scene, stream)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(e1.ev, stream));
    CUDA_TRY(cudaEventSynchronize(e1.ev));
    if (ms_device) CUDA_TRY(cudaEventElapsedTime(ms_device, e0.ev, e1.ev));
    for (uint32_t j = 0; j < edit->n_spheres; ++j) scene->sphere_material[edit->sphere_index[j]] = edit->spheres[j].material;
    for (uint32_t j = 0; j < edit->n_materials; ++j) scene->material_kind[edit->material_index[j]] = edit->materials[j].kind;
    rtd::find_lights(scene);
    return RT_OK;
}
RT_API_CATCH
