// rt_multi.cu — multi-GPU entries of the C-ABI (include/rt_api.h, SURVEY.md 8e): samples per pixel are split across
// the GPUs of one box, every GPU renders its samples of EVERY pixel into its own float4 accumulator, and the accumulators
// are summed and finalised by ONE fused kernel per GPU that reads the peers' accumulators over NVLink (k_reduce_tonemap,
// rt_kernels.cu) — each GPU reduces a band of rows and writes it straight into the root's image.  No NCCL call: the path has
// no other exchange step.
//
// Two hosts for the same data plane:
//  * rt_group_*  one PROCESS per GPU (torchrun, MPI, ...).  The accumulator, the barrier flags and the root's image are plain
//                cudaMalloc allocations exported as CUDA IPC handles; the caller moves the RT_GROUP_HANDLE_BYTES blobs between the
//                processes with whatever it has (torch.distributed.all_gather in bench.py).  Ordering between the GPUs is a
//                flag barrier in peer memory (one tiny kernel: release-store the epoch into every peer's flag word, acquire-spin on
//                one's own); every rank runs on its own GPU, so the spinning kernels are co-resident by construction.
//  * rt_multi_*  ONE process, N devices (what the reference's main(), main.cu:368-509, would become): a context per device,
//                cudaDeviceEnablePeerAccess, one host thread per device for the render, CUDA events for the cross-device ordering.
#include <atomic>
#include <chrono>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "rt_internal.hpp"

namespace {

constexpr int kMaxRanks = 16;     // PeerPtrs of k_reduce_tonemap
constexpr size_t kFlagBytes = 256; // kMaxRanks epoch words + the time-out flag, in their own 256-byte tail of the accumulator

size_t accum_bytes(int32_t w, int32_t h) { return (size_t(w) * size_t(h) * sizeof(float4) + 255u) & ~size_t(255); }

// Flag barrier over peer memory.  Thread r of the single CTA publishes `epoch` in rank r's flag word of THIS rank
// (a store over NVLink, release at system scope: everything this GPU wrote before — its accumulator, its band of the image —
// is visible to whoever acquires the flag) and then waits until rank r has done the same here.  Epochs only grow, so the
// words are never reset.  A peer that never arrives (a crashed process) must not wedge the GPU: after `spin_limit` polls the
// kernel gives up and raises flags[kMaxRanks], which the host turns into RT_ERR_CUDA.
struct PeerFlags {
    uint32_t* p[kMaxRanks];
};
__global__ void k_group_barrier(const __grid_constant__ PeerFlags peers, int rank, int world, uint32_t epoch, unsigned long long spin_limit) {
    const int r = int(threadIdx.x);
    if (r >= world) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(peers.p[r] + rank), "r"(epoch) : "memory");
    const uint32_t* mine = peers.p[rank] + r;
    uint32_t seen = 0;
    unsigned long long polls = 0;
    do {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(mine) : "memory");
        if (int32_t(seen - epoch) >= 0) break;
        __nanosleep(64);
    } while (++polls < spin_limit);
    if (int32_t(seen - epoch) < 0) atomicExch(peers.p[rank] + kMaxRanks, 1u);
    __threadfence_system();
}

} // namespace

// ------------------------------------------------------------------------------------------------ sharding ----
extern "C" rt_status rt_shard_samples(int32_t spp_total, int32_t rank, int32_t world, int32_t* first, int32_t* count) {
    ARG_CHECK(world >= 1 && rank >= 0 && rank < world && spp_total >= 0, "bad rank / world / spp_total");
    ARG_CHECK(first && count, "first/count is NULL");
    const int32_t base = spp_total / world, rem = spp_total % world;
    *count = base + (rank < rem ? 1 : 0);
    *first = rank * base + (rank < rem ? rank : rem);
    return RT_OK;
}

extern "C" rt_status rt_shard_rows(int32_t height, int32_t rank, int32_t world, int32_t* row_begin, int32_t* row_end) {
    ARG_CHECK(world >= 1 && rank >= 0 && rank < world && height >= 0, "bad rank / world / height");
    ARG_CHECK(row_begin && row_end, "row_begin/row_end is NULL");
    *row_begin = int32_t(int64_t(rank) * height / world);
    *row_end = int32_t(int64_t(rank + 1) * height / world);
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------ rt_group ----
struct rt_group {
    rt_context* ctx = nullptr;
    int32_t rank = 0, world = 1, width = 0, height = 0;
    void* accum = nullptr;  // [accum_bytes] float4 accumulator + kFlagBytes of flags (one allocation: one IPC handle)
    void* image = nullptr;  // root only: W*H*3 floats, then W*H*3 bytes
    void* peer_accum[kMaxRanks] = {};
    void* root_image = nullptr;
    bool opened[kMaxRanks] = {};
    bool opened_image = false;
    bool connected = false;
    uint32_t epoch = 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
};

namespace {
struct GroupHandle { // what rt_group_export writes (RT_GROUP_HANDLE_BYTES)
    uint32_t magic, rank, world, device;
    int32_t width, height;
    uint32_t has_image, pad;
    cudaIpcMemHandle_t accum, image;
};
static_assert(sizeof(GroupHandle) <= RT_GROUP_HANDLE_BYTES, "RT_GROUP_HANDLE_BYTES too small");
constexpr uint32_t kMagic = 0x52544750u; // "RTGP"

float* image_rgb(void* image) { return static_cast<float*>(image); }
uint8_t* image_rgb8(void* image, int32_t w, int32_t h) { return static_cast<uint8_t*>(image) + size_t(w) * h * 3 * sizeof(float); }

rt_status group_barrier(rt_group* g) {
    PeerFlags pf{};
    for (int r = 0; r < g->world; ++r) pf.p[r] = reinterpret_cast<uint32_t*>(static_cast<char*>(g->peer_accum[r]) + accum_bytes(g->width, g->height));
    ++g->epoch;
    // ~64 ns per poll: 2^27 polls are several seconds, far beyond any frame's skew between ranks
    k_group_barrier<<<1, 32, 0, g->ctx->stream>>>(pf, g->rank, g->world, g->epoch, 1ull << 27);
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}
} // namespace

extern "C" rt_status rt_group_create(rt_context* ctx, int32_t rank, int32_t world, int32_t width, int32_t height, rt_group** out) try {
    ARG_CHECK(ctx && out, "ctx/out is NULL");
    *out = nullptr;
    ARG_CHECK(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, "rank/world out of range (at most 16 ranks)");
    ARG_CHECK(width > 0 && height > 0 && uint64_t(width) * uint64_t(height) < (1ull << 31), "bad frame size");
    CUDA_TRY(cudaSetDevice(ctx->device));
    rt_group* g = new rt_group();
    g->ctx = ctx;
    g->rank = rank;
    g->world = world;
    g->width = width;
    g->height = height;
    const rt_status st = [&]() -> rt_status {
        const size_t ab = accum_bytes(width, height);
        CUDA_TRY(cudaMalloc(&g->accum, ab + kFlagBytes)); // cudaMalloc, not the pool: IPC-exportable
        CUDA_TRY(cudaMemsetAsync(g->accum, 0, ab + kFlagBytes, ctx->stream));
        if (rank == 0) CUDA_TRY(cudaMalloc(&g->image, size_t(width) * height * (3 * sizeof(float) + 3)));
        for (auto& e : g->ev) CUDA_TRY(cudaEventCreate(&e));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        g->peer_accum[rank] = g->accum;
        if (rank == 0) g->root_image = g->image;
        if (world == 1) g->connected = true;
        return RT_OK;
    }();
    if (st != RT_OK) {
        rt_group_destroy(g);
        return st;
    }
    *out = g;
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_group_export(const rt_group* g, void* handle) try {
    ARG_CHECK(g && handle, "group/handle is NULL");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    GroupHandle h{};
    h.magic = kMagic;
    h.rank = uint32_t(g->rank);
    h.world = uint32_t(g->world);
    h.device = uint32_t(g->ctx->device);
    h.width = g->width;
    h.height = g->height;
    h.has_image = g->image ? 1u : 0u;
    CUDA_TRY(cudaIpcGetMemHandle(&h.accum, g->accum));
    if (g->image) CUDA_TRY(cudaIpcGetMemHandle(&h.image, g->image));
    memset(handle, 0, RT_GROUP_HANDLE_BYTES);
    memcpy(handle, &h, sizeof h);
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_group_connect(rt_group* g, const void* handles) try {
    ARG_CHECK(g && handles, "group/handles is NULL");
    ARG_CHECK(!g->connected || g->world == 1, "group is already connected");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    const char* base = static_cast<const char*>(handles);
    for (int r = 0; r < g->world; ++r) {
        GroupHandle h;
        memcpy(&h, base + size_t(r) * RT_GROUP_HANDLE_BYTES, sizeof h);
        ARG_CHECK(h.magic == kMagic && int32_t(h.rank) == r && int32_t(h.world) == g->world, "handle table is not in rank order / from another group");
        ARG_CHECK(h.width == g->width && h.height == g->height, "ranks disagree about the frame size");
        if (r != g->rank) {
            CUDA_TRY(cudaIpcOpenMemHandle(&g->peer_accum[r], h.accum, cudaIpcMemLazyEnablePeerAccess));
            g->opened[r] = true;
        }
        if (r == 0 && g->rank != 0) {
            ARG_CHECK(h.has_image != 0u, "rank 0 exported no image");
            CUDA_TRY(cudaIpcOpenMemHandle(&g->root_image, h.image, cudaIpcMemLazyEnablePeerAccess));
            g->opened_image = true;
        }
    }
    g->connected = true;
    return RT_OK;
}
RT_API_CATCH

extern "C" void* rt_group_accum(const rt_group* g) { return g ? g->accum : nullptr; }

extern "C" rt_status rt_group_begin_frame(rt_group* g) try {
    ARG_CHECK(g && g->connected, "group is NULL / not connected");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    // (ordered after the closing barrier of the previous frame: no peer still reads this accumulator)
    CUDA_TRY(cudaMemsetAsync(g->accum, 0, size_t(g->width) * g->height * sizeof(float4), g->ctx->stream));
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_group_finish_frame(rt_group* g, int32_t want_rgb8, float* ms_reduce) try {
    ARG_CHECK(g && g->connected, "group is NULL / not connected");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    cudaStream_t st = g->ctx->stream;
    rt_status s = RT_OK;
    if (ms_reduce) CUDA_TRY(cudaEventRecord(g->ev[0], st));
    if (g->world > 1 && (s = group_barrier(g)) != RT_OK) return s; // every rank's accumulator is complete
    int32_t r0 = 0, r1 = 0;
    rt_shard_rows(g->height, g->rank, g->world, &r0, &r1);
    rtd::launch_reduce_tonemap(g->peer_accum, g->world, nullptr, g->width, g->height, r0, r1, image_rgb(g->root_image),
                               want_rgb8 ? image_rgb8(g->root_image, g->width, g->height) : nullptr, nullptr, g->ctx->sm_count, st);
    CUDA_TRY(cudaGetLastError());
    if (g->world > 1 && (s = group_barrier(g)) != RT_OK) return s; // every band is in the root's image; accumulators are free again
    if (ms_reduce) {
        CUDA_TRY(cudaEventRecord(g->ev[1], st));
        CUDA_TRY(cudaEventSynchronize(g->ev[1]));
        CUDA_TRY(cudaEventElapsedTime(ms_reduce, g->ev[0], g->ev[1]));
    }
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_group_read_frame(rt_group* g, float* out_rgb, uint8_t* out_rgb8) try {
    ARG_CHECK(g && g->connected, "group is NULL / not connected");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    cudaStream_t st = g->ctx->stream;
    const size_t npix = size_t(g->width) * g->height;
    if (g->rank == 0) {
        if (out_rgb) CUDA_TRY(cudaMemcpyAsync(out_rgb, image_rgb(g->image), npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (out_rgb8) CUDA_TRY(cudaMemcpyAsync(out_rgb8, image_rgb8(g->image, g->width, g->height), npix * 3, cudaMemcpyDeviceToHost, st));
    }
    uint32_t timed_out = 0;
    CUDA_TRY(cudaMemcpyAsync(&timed_out, static_cast<char*>(g->accum) + accum_bytes(g->width, g->height) + kMaxRanks * sizeof(uint32_t),
                          sizeof timed_out, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (timed_out) {
        rtd::set_error("rt_group: a peer never reached the barrier (rank %d gave up waiting)", g->rank);
        return RT_ERR_CUDA;
    }
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_group_read_accum(rt_group* g, float* out_accum) try {
    ARG_CHECK(g && out_accum, "group/out is NULL");
    CUDA_TRY(cudaSetDevice(g->ctx->device));
    CUDA_TRY(cudaMemcpyAsync(out_accum, g->accum, size_t(g->width) * g->height * sizeof(float4), cudaMemcpyDeviceToHost, g->ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(g->ctx->stream));
    return RT_OK;
}
RT_API_CATCH

extern "C" void rt_group_destroy(rt_group* g) {
    if (!g) return;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->ctx->stream);
    for (int r = 0; r < kMaxRanks; ++r)
        if (g->opened[r] && g->peer_accum[r]) cudaIpcCloseMemHandle(g->peer_accum[r]);
    if (g->opened_image && g->root_image) cudaIpcCloseMemHandle(g->root_image);
    if (g->accum) cudaFree(g->accum);
    if (g->image) cudaFree(g->image);
    for (auto& e : g->ev)
        if (e) cudaEventDestroy(e);
    delete g;
}

// ------------------------------------------------------------------------------------------------ rt_multi ----
struct rt_multi {
    int32_t n = 0;
    std::vector<rt_context*> ctx;
    std::vector<rt_scene*> scene;
    std::vector<void*> accum; // per device, sized for the largest frame rendered so far
    size_t accum_px = 0;
    void* image = nullptr;    // device 0: W*H*3 floats + W*H*3 bytes
    size_t image_px = 0;
    std::vector<cudaEvent_t> ev_done, ev_red;
    cudaEvent_t ev_t[2] = {nullptr, nullptr};
};

extern "C" rt_status rt_multi_create(const int32_t* devices, int32_t n_devices, rt_multi** out) try {
    ARG_CHECK(out, "out is NULL");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        rtd::set_error("no CUDA device available; this library has no CPU fallback");
        return RT_ERR_NO_DEVICE;
    }
    if (n_devices <= 0) n_devices = count; // all of them
    ARG_CHECK(n_devices <= kMaxRanks && n_devices <= count, "more devices requested than present (or than 16)");
    rt_multi* m = new rt_multi();
    m->n = n_devices;
    const rt_status st = [&]() -> rt_status {
        for (int k = 0; k < n_devices; ++k) {
            const int dev = devices ? devices[k] : k;
            for (int j = 0; j < k; ++j) ARG_CHECK(m->ctx[j]->device != dev, "device listed twice");
            rt_context* c = nullptr;
            const rt_status s = rt_context_create(dev, &c);
            if (s != RT_OK) return s;
            m->ctx.push_back(c);
        }
        for (int a = 0; a < n_devices; ++a) { // every device reads every other device's accumulator; all write device 0's image
            CUDA_TRY(cudaSetDevice(m->ctx[a]->device));
            for (int b = 0; b < n_devices; ++b) {
                if (a == b) continue;
                int can = 0;
                CUDA_TRY(cudaDeviceCanAccessPeer(&can, m->ctx[a]->device, m->ctx[b]->device));
                if (!can) {
                    rtd::set_error("device %d cannot access device %d's memory (no NVLink / P2P path)", m->ctx[a]->device, m->ctx[b]->device);
                    return RT_ERR_UNSUPPORTED;
                }
                const cudaError_t e = cudaDeviceEnablePeerAccess(m->ctx[b]->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CUDA_TRY(e);
                cudaGetLastError();
            }
        }
        m->scene.assign(n_devices, nullptr);
        m->accum.assign(n_devices, nullptr);
        m->ev_done.assign(n_devices, nullptr);
        m->ev_red.assign(n_devices, nullptr);
        for (int k = 0; k < n_devices; ++k) {
            CUDA_TRY(cudaSetDevice(m->ctx[k]->device));
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_done[k], cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&m->ev_red[k], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
        for (auto& e : m->ev_t) CUDA_TRY(cudaEventCreate(&e));
        return RT_OK;
    }();
    if (st != RT_OK) {
        rt_multi_destroy(m);
        return st;
    }
    *out = m;
    return RT_OK;
}
RT_API_CATCH

extern "C" int32_t rt_multi_size(const rt_multi* m) { return m ? m->n : 0; }

namespace {
// call(k) for every member k, side by side on one host thread each; the first failing member's status, with its device
// in the message
template <class Call>
rt_status each_member(rt_multi* m, Call&& call) {
    std::vector<rt_status> st(m->n, RT_OK);
    std::vector<std::string> msg(m->n);
    std::vector<std::thread> th;
    for (int k = 0; k < m->n; ++k)
        th.emplace_back([&, k] {
            st[k] = call(k);
            if (st[k] != RT_OK) msg[k] = rt_last_error();
        });
    for (auto& t : th) t.join();
    for (int k = 0; k < m->n; ++k)
        if (st[k] != RT_OK) {
            rtd::set_error("device %d: %s", m->ctx[k]->device, msg[k].c_str());
            return st[k];
        }
    return RT_OK;
}
} // namespace

extern "C" rt_status rt_multi_set_scene(rt_multi* m, const rt_scene_desc* desc) try {
    ARG_CHECK(m && desc, "multi/desc is NULL");
    return each_member(m, [&](int k) { // uploads + BVH builds of the devices run side by side
        if (m->scene[k]) rt_scene_destroy(m->scene[k]);
        m->scene[k] = nullptr;
        return rt_scene_create(m->ctx[k], desc, &m->scene[k]);
    });
}
RT_API_CATCH

extern "C" rt_status rt_multi_update_scene(rt_multi* m, const rt_scene_edit* edit) try {
    ARG_CHECK(m && edit, "multi/edit is NULL");
    for (int k = 0; k < m->n; ++k) ARG_CHECK(m->scene[k] != nullptr, "no scene: call rt_multi_set_scene first");
    return each_member(m, [&](int k) { return rt_scene_update(m->ctx[k], m->scene[k], edit, nullptr); });
}
RT_API_CATCH

extern "C" rt_status rt_multi_render(rt_multi* m, const rt_render_params* p, float* out_rgb, uint8_t* out_rgb8, rt_stats* stats,
                                     float* ms_reduce) try {
    ARG_CHECK(m && p, "multi/params is NULL");
    ARG_CHECK(out_rgb || out_rgb8, "no output buffer");
    ARG_CHECK(p->width > 0 && p->height > 0 && uint64_t(p->width) * uint64_t(p->height) < (1ull << 31), "bad frame size");
    for (int k = 0; k < m->n; ++k) ARG_CHECK(m->scene[k] != nullptr, "no scene: call rt_multi_set_scene first");
    const size_t npix = size_t(p->width) * p->height;
    if (m->accum_px < npix) {
        for (int k = 0; k < m->n; ++k) {
            CUDA_TRY(cudaSetDevice(m->ctx[k]->device));
            if (m->accum[k]) cudaFree(m->accum[k]);
            m->accum[k] = nullptr;
            CUDA_TRY(cudaMalloc(&m->accum[k], npix * sizeof(float4)));
        }
        m->accum_px = npix;
    }
    if (m->image_px < npix) {
        CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
        if (m->image) cudaFree(m->image);
        m->image = nullptr;
        CUDA_TRY(cudaMalloc(&m->image, npix * (3 * sizeof(float) + 3)));
        m->image_px = npix;
    }
    // ---- render: one host thread per device (the wavefront loop polls its queue counters) ----
    std::vector<rt_status> st(m->n, RT_OK);
    std::vector<std::string> msg(m->n);
    std::vector<rt_stats> rs(m->n);
    std::vector<std::thread> th;
    const auto t0 = std::chrono::steady_clock::now();
    for (int k = 0; k < m->n; ++k)
        th.emplace_back([&, k] {
            rt_render_params q = *p;
            int32_t first = 0, count = 0;
            rt_shard_samples(p->spp, k, m->n, &first, &count);
            q.spp = count;
            q.sample_offset = p->sample_offset + first;
            cudaSetDevice(m->ctx[k]->device);
            cudaError_t e = cudaMemsetAsync(m->accum[k], 0, npix * sizeof(float4), m->ctx[k]->stream);
            if (e == cudaSuccess) st[k] = rt_render_accum_device(m->ctx[k], m->scene[k], &q, m->accum[k], &rs[k]);
            else st[k] = RT_ERR_CUDA;
            if (st[k] != RT_OK) msg[k] = e == cudaSuccess ? rt_last_error() : cudaGetErrorString(e);
            else cudaEventRecord(m->ev_done[k], m->ctx[k]->stream);
        });
    for (auto& t : th) t.join();
    for (int k = 0; k < m->n; ++k)
        if (st[k] != RT_OK) {
            rtd::set_error("device %d: %s", m->ctx[k]->device, msg[k].c_str());
            return st[k];
        }
    // ---- fused reduce + finalisation: device k sums band k of all accumulators over NVLink into device 0's image ----
    void* peers[kMaxRanks] = {};
    for (int k = 0; k < m->n; ++k) peers[k] = m->accum[k];
    CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
    CUDA_TRY(cudaEventRecord(m->ev_t[0], m->ctx[0]->stream));
    for (int k = 0; k < m->n; ++k) {
        CUDA_TRY(cudaSetDevice(m->ctx[k]->device));
        cudaStream_t s = m->ctx[k]->stream;
        if (k == 0) CUDA_TRY(cudaStreamWaitEvent(s, m->ev_t[0], 0));
        for (int j = 0; j < m->n; ++j)
            if (j != k) CUDA_TRY(cudaStreamWaitEvent(s, m->ev_done[j], 0));
        int32_t r0 = 0, r1 = 0;
        rt_shard_rows(p->height, k, m->n, &r0, &r1);
        rtd::launch_reduce_tonemap(peers, m->n, nullptr, p->width, p->height, r0, r1, image_rgb(m->image),
                                   out_rgb8 ? image_rgb8(m->image, p->width, p->height) : nullptr, nullptr, m->ctx[k]->sm_count, s);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(m->ev_red[k], s));
    }
    CUDA_TRY(cudaSetDevice(m->ctx[0]->device));
    cudaStream_t s0 = m->ctx[0]->stream;
    for (int k = 1; k < m->n; ++k) CUDA_TRY(cudaStreamWaitEvent(s0, m->ev_red[k], 0));
    CUDA_TRY(cudaEventRecord(m->ev_t[1], s0));
    if (out_rgb) CUDA_TRY(cudaMemcpyAsync(out_rgb, image_rgb(m->image), npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, s0));
    if (out_rgb8) CUDA_TRY(cudaMemcpyAsync(out_rgb8, image_rgb8(m->image, p->width, p->height), npix * 3, cudaMemcpyDeviceToHost, s0));
    CUDA_TRY(cudaStreamSynchronize(s0));
    float red = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&red, m->ev_t[0], m->ev_t[1]));
    if (ms_reduce) *ms_reduce = red;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->paths = uint64_t(npix) * uint64_t(p->spp);
        for (int k = 0; k < m->n; ++k) {
            stats->rays += rs[k].rays;
            stats->launches += rs[k].launches;
            if (rs[k].ms_total > stats->ms_total) stats->ms_total = rs[k].ms_total; // slowest device
            if (rs[k].iterations > stats->iterations) stats->iterations = rs[k].iterations;
        }
        stats->launches += uint32_t(m->n);
        stats->ms_tonemap = red;
        stats->ms_d2h = float(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count()); // wall clock of the call
    }
    return RT_OK;
}
RT_API_CATCH

extern "C" rt_status rt_multi_read_accum(rt_multi* m, int32_t member, float* out_accum) try {
    ARG_CHECK(m && out_accum && member >= 0 && member < m->n && m->accum[member], "bad member / no frame rendered yet");
    CUDA_TRY(cudaSetDevice(m->ctx[member]->device));
    CUDA_TRY(cudaMemcpyAsync(out_accum, m->accum[member], m->accum_px * sizeof(float4), cudaMemcpyDeviceToHost, m->ctx[member]->stream));
    CUDA_TRY(cudaStreamSynchronize(m->ctx[member]->stream));
    return RT_OK;
}
RT_API_CATCH

extern "C" void rt_multi_destroy(rt_multi* m) {
    if (!m) return;
    for (int k = 0; k < int(m->ctx.size()); ++k) {
        cudaSetDevice(m->ctx[k]->device);
        cudaStreamSynchronize(m->ctx[k]->stream);
        if (k < int(m->scene.size()) && m->scene[k]) rt_scene_destroy(m->scene[k]);
        if (k < int(m->accum.size()) && m->accum[k]) cudaFree(m->accum[k]);
        if (k < int(m->ev_done.size()) && m->ev_done[k]) cudaEventDestroy(m->ev_done[k]);
        if (k < int(m->ev_red.size()) && m->ev_red[k]) cudaEventDestroy(m->ev_red[k]);
    }
    if (!m->ctx.empty()) {
        cudaSetDevice(m->ctx[0]->device);
        if (m->image) cudaFree(m->image);
        for (auto& e : m->ev_t)
            if (e) cudaEventDestroy(e);
    }
    for (auto* c : m->ctx) rt_context_destroy(c);
    delete m;
}
