// rt_api.cu — C-ABI of librt_b200.so (include/rt_api.h): contexts, render / accumulate / probe / tonemap / JPEG / image
// entry points (scenes: rt_scene.cu).  Host logic only; the kernels live in rt_kernels.cu / rt_wavefront.cu / rt_lbvh.cu.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "rt_internal.hpp"
#include "rt_jpeg_decode.cuh"

namespace {
thread_local std::string g_last_error;
thread_local cudaMemPool_t g_thread_pool = nullptr;
} // namespace

namespace rtd {
void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
}
void set_error_message(const char* msg) { g_last_error = msg ? msg : ""; }
void set_thread_mempool(cudaMemPool_t pool) { g_thread_pool = pool; }
cudaError_t malloc_async_bytes(void** p, size_t bytes, cudaStream_t st) {
    return g_thread_pool ? cudaMallocFromPoolAsync(p, bytes, g_thread_pool, st) : cudaMallocAsync(p, bytes, st);
}
} // namespace rtd

using rtd::make_current;
using rtd::set_error;

namespace rtd {
// camera ctor (camera.h:7-31) in host float arithmetic
void make_camera(const rt_camera& c, DCamera& out) {
    auto V = [](const float* p) { return rtd::V3{p[0], p[1], p[2]}; };
    auto sub = [](rtd::V3 a, rtd::V3 b) { return rtd::V3{a.x - b.x, a.y - b.y, a.z - b.z}; };
    auto mul = [](rtd::V3 a, float s) { return rtd::V3{a.x * s, a.y * s, a.z * s}; };
    auto cross = [](rtd::V3 a, rtd::V3 b) {
        return rtd::V3{a.y * b.z - a.z * b.y, -(a.x * b.z - a.z * b.x), a.x * b.y - a.y * b.x};
    };
    auto norm = [](rtd::V3 a) {
        if (a.x == 0.f && a.y == 0.f && a.z == 0.f) return a;
        float l = std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z);
        return rtd::V3{a.x / l, a.y / l, a.z / l};
    };
    out.t0 = c.time0;
    out.t1 = c.time1;
    out.lens_radius = c.aperture / 2;
    float theta = float(c.vfov * M_PI / 180.f);
    float half_height = std::tan(theta / 2.f);
    float half_width = c.aspect * half_height;
    rtd::V3 lookfrom = V(c.lookfrom), lookat = V(c.lookat), up = V(c.up);
    out.origin = lookfrom;
    rtd::V3 w = norm(sub(lookfrom, lookat));
    rtd::V3 u = norm(cross(up, w));
    rtd::V3 v = cross(w, u);
    out.u = u;
    out.v = v;
    out.lower_left = sub(sub(sub(out.origin, mul(u, half_width * c.focus_dist)), mul(v, half_height * c.focus_dist)),
                         mul(w, c.focus_dist));
    out.horizontal = mul(u, 2 * half_width * c.focus_dist);
    out.vertical = mul(v, 2 * half_height * c.focus_dist);
}
} // namespace rtd
namespace {

rt_status check_params(const rt_render_params* p) {
    ARG_CHECK(p != nullptr, "params is NULL");
    ARG_CHECK(p->width > 0 && p->height > 0, "width/height must be positive");
    ARG_CHECK(p->spp >= 0 && p->sample_offset >= 0, "spp/sample_offset must be >= 0");
    ARG_CHECK(p->max_depth >= 0 && p->max_depth < (1 << 23), "max_depth out of range");
    ARG_CHECK(p->pipeline <= RT_PIPE_MEGAKERNEL, "bad pipeline");
    ARG_CHECK((p->flags & ~RT_RENDER_EMITTER_SAMPLING) == 0u, "unknown render flags");
    ARG_CHECK(std::isfinite(p->tmin) && std::isfinite(p->bloom) && std::isfinite(p->world[0]) && std::isfinite(p->world[1]) &&
                  std::isfinite(p->world[2]),
              "tmin / bloom / world colour is not finite");
    ARG_CHECK(uint64_t(p->width) * uint64_t(p->height) < (1ull << 31), "frame has more than 2^31 pixels");
    return RT_OK;
}

rtd::DRenderParams to_device_params(const rt_render_params& p) {
    rtd::DRenderParams d;
    d.div_width = rtd::make_fastdiv(uint32_t(p.width));
    d.div_npix = rtd::make_fastdiv(uint32_t(uint64_t(p.width) * uint64_t(p.height))); // < 2^32: check_params
    d.width = p.width;
    d.height = p.height;
    d.spp = p.spp;
    d.sample_offset = p.sample_offset;
    d.max_depth = p.max_depth;
    d.seed = p.seed;
    d.tmin = p.tmin;
    d.world_r = p.world[0];
    d.world_g = p.world[1];
    d.world_b = p.world[2];
    d.bloom = p.bloom;
    d.flags = p.flags;
    d.adapt_pixels = nullptr;
    d.adapt_first = 0;
    d.adapt_plane = 0;
    d.frame_cams = nullptr;
    d.div_spp = rtd::make_fastdiv(1u);
    return d;
}

// a context buffer of at least n elements (it grows, never shrinks)
template <class T>
rt_status grow(T*& p, size_t& cap, size_t n) {
    if (cap < n) {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        CUDA_TRY(cudaMalloc(&p, n * sizeof(T)));
        cap = n;
    }
    return RT_OK;
}

rt_status ensure_jpeg(rt_context* ctx) {
    if (!ctx->jpg) {
        ctx->jpg = rtd::jpeg_create();
        if (!ctx->jpg) {
            set_error("jpeg_create failed: %s", cudaGetErrorString(cudaGetLastError()));
            return RT_ERR_OOM;
        }
    }
    return RT_OK;
}

rt_status jpeg_from_device(rt_context* ctx, const uint8_t* rgb8_dev, int32_t w, int32_t h, int32_t quality, uint8_t* out, size_t cap,
                           size_t* n_bytes, float* ms_device) {
    rt_status st = ensure_jpeg(ctx);
    if (st != RT_OK) return st;
    size_t n = 0;
    cudaError_t e = rtd::jpeg_encode(ctx->jpg, rgb8_dev, w, h, quality, out, cap, &n, ctx->stream, ms_device);
    if (n_bytes) *n_bytes = n;
    if (e == cudaErrorInvalidValue && out && n > cap) {
        set_error("JPEG needs %zu bytes, the output buffer holds %zu", n, cap);
        return RT_ERR_INVALID_ARG;
    }
    if (e != cudaSuccess) {
        set_error("jpeg_encode: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA;
    }
    return RT_OK;
}

// One render pass: rp.spp samples of every pixel (of the rp.adapt_pixels list when it is set) added into accum (device);
// rays are added to ctx->d_ray_counter.
rt_status render_pass(rt_context* ctx, const rt_scene* scene, const rtd::DRenderParams& rp, uint32_t pipeline_param, float4* accum,
                      uint32_t* launches_out, uint32_t* iterations_out) {
    const bool use_bvh = scene->d.nodes != nullptr;
    uint32_t pipeline = pipeline_param == RT_PIPE_AUTO ? uint32_t(RT_PIPE_WAVEFRONT) : pipeline_param;
    uint32_t launches = 0, iterations = 0;
    if (pipeline == RT_PIPE_MEGAKERNEL) {
        rtd::launch_render_mega(scene->d, rp, use_bvh, accum, ctx->d_ray_counter, ctx->sm_count, ctx->stream);
        launches = 1;
        iterations = 1;
    } else {
        const size_t npix = rp.adapt_pixels ? size_t(rp.div_npix.d) : size_t(rp.width) * size_t(rp.height);
        const size_t npaths = npix * size_t(rp.spp);
        // pool of path slots (RT_WF_POOL overrides).  Measured on C1 (ms/frame): 256 Ki 18.7, 512 Ki 14.7, 1 Mi 13.5,
        // 2 Mi 12.6, 4 Mi 12.4 (before the later kernel work), then 4 Mi 11.0, 8 Mi 11.0, 16 Mi 10.5 — fewer, fuller
        // iterations beat keeping the 64-byte records L2-resident.  16 Mi slots = 1 GiB of records + 1 GiB of queues.
        size_t pool_cap = size_t(16) << 20;
        if (const char* e = getenv("RT_WF_POOL")) {
            long long v = atoll(e);
            if (v >= 1024 && v <= (1ll << 28)) pool_cap = size_t(v);
        }
        size_t pool = npaths < pool_cap ? npaths : pool_cap;
        if (pool < 1024) pool = 1024;
        if (!ctx->wf || rtd::wavefront_pool(ctx->wf) < pool) {
            if (ctx->wf) rtd::wavefront_destroy(ctx->wf);
            ctx->wf = rtd::wavefront_create(pool, ctx->stream);
            if (!ctx->wf) {
                set_error("wavefront_create(%zu paths) failed: %s", pool, cudaGetErrorString(cudaGetLastError()));
                return RT_ERR_OOM;
            }
        }
        if (!rtd::wavefront_render(ctx->wf, scene->d, rp, use_bvh, accum, ctx->d_ray_counter, ctx->sm_count, ctx->stream, &launches,
                                   &iterations)) {
            const cudaError_t e = cudaGetLastError();
            set_error("wavefront_render: frame unfinished after %u iterations (%s)", iterations, cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
    }
    CUDA_TRY(cudaGetLastError());
    *launches_out = launches;
    *iterations_out = iterations;
    return RT_OK;
}

// The timed window of a render when stats are wanted: stats_begin zeroes the ray counter and records ev[0]; stats_end
// records ev[1], reads the counter back (synchronising) and fills the render's part of *stats.
rt_status stats_begin(rt_context* ctx, const rt_stats* stats) {
    if (!stats) return RT_OK;
    CUDA_TRY(cudaMemsetAsync(ctx->d_ray_counter, 0, sizeof(unsigned long long), ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[0], ctx->stream));
    return RT_OK;
}

rt_status stats_end(rt_context* ctx, rt_stats* stats, uint64_t paths, uint32_t launches, uint32_t iterations) {
    if (!stats) return RT_OK;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    unsigned long long rays = 0;
    CUDA_TRY(cudaMemcpyAsync(&rays, ctx->d_ray_counter, sizeof rays, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    memset(stats, 0, sizeof *stats);
    CUDA_TRY(cudaEventElapsedTime(&stats->ms_total, ctx->ev[0], ctx->ev[1]));
    stats->paths = paths;
    stats->rays = rays;
    stats->launches = launches;
    stats->iterations = iterations;
    return RT_OK;
}

// Core: adds rp.spp samples per pixel into accum (device).  Fills stats if requested
// (which synchronises the stream).
rt_status render_rp(rt_context* ctx, const rt_scene* scene, const rtd::DRenderParams& rp, uint32_t pipeline, float4* accum,
                    rt_stats* stats) {
    uint32_t launches = 0, iterations = 0;
    rt_status st = stats_begin(ctx, stats);
    if (st != RT_OK) return st;
    if ((st = render_pass(ctx, scene, rp, pipeline, accum, &launches, &iterations)) != RT_OK) return st;
    return stats_end(ctx, stats, uint64_t(rp.width) * uint64_t(rp.height) * uint64_t(rp.spp), launches, iterations);
}

// the pixel finalisation of the n_frames frames of ctx->accum into ctx->out_rgb
rt_status tonemap_frames(rt_context* ctx, const rt_render_params* p, int32_t n_frames) {
    const size_t npix = size_t(p->width) * size_t(p->height);
    for (int32_t f = 0; f < n_frames; ++f)
        rtd::launch_tonemap(ctx->accum + size_t(f) * npix, p->width, p->height, ctx->out_rgb + size_t(f) * npix * 3, nullptr,
                            ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

struct HostCopy {
    const void* src = nullptr;
    void* dst = nullptr;
    size_t bytes = 0;
};

// The end of a host render entry, after the render into ctx->accum: `finalise` (the kernels that make the device image;
// nullptr: none) between ev[1] and ev[2], the copy of `image` to the host between ev[2] and ev[3], then `also` (untimed),
// one synchronisation, and the two windows in stats->ms_tonemap / ms_d2h.  *out_stats = stats on success.
template <class Finalise>
rt_status finish_to_host(rt_context* ctx, Finalise&& finalise, const HostCopy& image, rt_stats& stats, rt_stats* out_stats,
                         const HostCopy& also = {}) {
    constexpr bool kFinalise = !std::is_null_pointer<std::decay_t<Finalise>>::value;
    if constexpr (kFinalise) {
        CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
        const rt_status st = finalise();
        if (st != RT_OK) return st;
    }
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(image.dst, image.src, image.bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    if (also.bytes) CUDA_TRY(cudaMemcpyAsync(also.dst, also.src, also.bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if constexpr (kFinalise) CUDA_TRY(cudaEventElapsedTime(&stats.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&stats.ms_d2h, ctx->ev[2], ctx->ev[3]));
    if (out_stats) *out_stats = stats;
    return RT_OK;
}

} // namespace

extern "C" {

int rt_api_version(void) { return RT_API_VERSION; }

const char* rt_last_error(void) { return g_last_error.c_str(); }

void rt_default_render_params(rt_render_params* p) {
    if (!p) return;
    memset(p, 0, sizeof *p);
    p->width = 1200;  // common.h:13
    p->height = 600;  // common.h:14
    p->spp = 100;     // main.cu:15
    p->sample_offset = 0;
    p->max_depth = 50; // common.h:19
    p->seed = 1000;    // common.h:20
    p->tmin = 0.00001f; // main.cu:45
    p->world[0] = 1.f;  // main.cu:40
    p->world[1] = .8f;
    p->world[2] = .7f;
    p->bloom = 0.1f; // main.cu:49
    p->pipeline = RT_PIPE_AUTO;
    p->flags = 0; // the reference's estimator
}

rt_status rt_context_create(int device, rt_context** out) try {
    ARG_CHECK(out != nullptr, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
        cudaGetLastError();
        return RT_ERR_NO_DEVICE;
    }
    ARG_CHECK(device >= 0 && device < count, "device index out of range");
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; librt_b200 carries sm_100a code only", device, prop.major, prop.minor);
        return RT_ERR_UNSUPPORTED;
    }
    rt_context* ctx = new (std::nothrow) rt_context();
    if (!ctx) return RT_ERR_OOM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    // everything created below is released by rt_context_destroy when a later step fails
    const rt_status st = [&]() -> rt_status {
        CUDA_TRY(cudaSetDevice(device));
        CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        // A memory pool of the context's own for scene data: freed scene memory stays in it (release threshold = max)
        // instead of going back to the driver, without touching the device's DEFAULT pool, which torch and every other
        // user of cudaMallocAsync in the process share.
        cudaMemPoolProps pp{};
        pp.allocType = cudaMemAllocationTypePinned;
        pp.handleTypes = cudaMemHandleTypeNone;
        pp.location.type = cudaMemLocationTypeDevice;
        pp.location.id = device;
        CUDA_TRY(cudaMemPoolCreate(&ctx->pool, &pp));
        unsigned long long keep = ~0ull;
        CUDA_TRY(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
        CUDA_TRY(cudaMalloc(&ctx->d_ray_counter, sizeof(unsigned long long)));
        for (auto& ev : ctx->ev) CUDA_TRY(cudaEventCreate(&ev));
        return RT_OK;
    }();
    if (st != RT_OK) {
        rt_context_destroy(ctx);
        return st;
    }
    *out = ctx;
    return RT_OK;
} RT_API_CATCH

void rt_context_destroy(rt_context* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream); // polling copies of the last render may still be in flight
    if (ctx->wf) rtd::wavefront_destroy(ctx->wf);
    if (ctx->jpg) rtd::jpeg_destroy(ctx->jpg);
    if (ctx->rgb8) cudaFree(ctx->rgb8);
    if (ctx->accum) cudaFree(ctx->accum);
    if (ctx->out_rgb) cudaFree(ctx->out_rgb);
    if (ctx->d_ray_counter) cudaFree(ctx->d_ray_counter);
    for (auto& c : ctx->array_cache) cudaFreeArray(c.arr);
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

rt_status rt_context_set_stream(rt_context* ctx, void* cuda_stream) try {
    ARG_CHECK(ctx != nullptr, "ctx is NULL");
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = static_cast<cudaStream_t>(cuda_stream);
    ctx->own_stream = false;
    return RT_OK;
} RT_API_CATCH

rt_status rt_context_synchronize(rt_context* ctx) try {
    ARG_CHECK(ctx != nullptr, "ctx is NULL");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
} RT_API_CATCH

rt_status rt_trace_primary(rt_context* ctx, const rt_scene* scene, const rt_ray* rays, size_t n, float tmin, int use_bvh,
                           rt_hit* hits) try {
    ARG_CHECK(ctx && scene, "ctx/scene is NULL");
    ARG_CHECK(n == 0 || (rays && hits), "rays/hits is NULL");
    ARG_CHECK(use_bvh >= 0 && use_bvh <= 3, "use_bvh must be 0 (list), 1 (BVH), 2 (4-wide BVH) or 3 (quantised 4-wide BVH)");
    ARG_CHECK(use_bvh != 2 || scene->d.nodes4 != nullptr, "use_bvh = 2: the scene has no 4-wide nodes");
    ARG_CHECK(use_bvh != 3 || scene->d.nodes4q != nullptr, "use_bvh = 3: the scene has no quantised 4-wide nodes");
    if (n == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::PoolBuffer<rt_ray> d_rays;
    rtd::PoolBuffer<rt_hit> d_hits;
    CUDA_TRY(d_rays.alloc(n, ctx->stream));
    cudaError_t e = d_hits.alloc(n, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rays.get(), rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::launch_trace_primary(scene->d, d_rays.get(), n, tmin, use_bvh, d_hits.get(), ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hits, d_hits.get(), n * sizeof(rt_hit), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("rt_trace_primary: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    return RT_OK;
} RT_API_CATCH

rt_status rt_shade_probe(rt_context* ctx, const rt_scene* scene, const rt_ray* rays, size_t n, const rt_render_params* p,
                         int use_bvh, rt_shade_sample* out) try {
    ARG_CHECK(ctx && scene && p, "ctx/scene/params is NULL");
    ARG_CHECK(n == 0 || (rays && out), "rays/out is NULL");
    ARG_CHECK(n < (size_t(1) << 32), "too many rays (the Philox key holds a 32-bit ray index)");
    if (n == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::PoolBuffer<rt_ray> d_rays;
    rtd::PoolBuffer<rt_shade_sample> d_out;
    CUDA_TRY(d_rays.alloc(n, ctx->stream));
    cudaError_t e = d_out.alloc(n, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rays.get(), rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::DRenderParams rp = to_device_params(*p);
        rp.flags = 0; // the probe reports the reference estimator's terms (rt_shade_sample carries no path weight)
        rtd::launch_shade_probe(scene->d, rp, d_rays.get(), n, use_bvh != 0, d_out.get(), ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out.get(), n * sizeof(rt_shade_sample), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("rt_shade_probe: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    return RT_OK;
} RT_API_CATCH

rt_status rt_render_accum_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, void* accum_dev,
                                 rt_stats* stats) try {
    ARG_CHECK(ctx && scene && accum_dev, "ctx/scene/accum_dev is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    return render_rp(ctx, scene, to_device_params(*p), p->pipeline, static_cast<float4*>(accum_dev), stats);
} RT_API_CATCH

rt_status rt_render_accum(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, float* out_accum, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_accum, "ctx/scene/out_accum is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_rp(ctx, scene, to_device_params(*p), p->pipeline, ctx->accum, &local)) != RT_OK) return st;
    return finish_to_host(ctx, nullptr, {ctx->accum, out_accum, npix * sizeof(float4)}, local, stats);
} RT_API_CATCH

rt_status rt_tonemap_device(rt_context* ctx, const void* accum_dev, int32_t width, int32_t height, void* out_rgb_dev,
                            void* out_rgb8_dev) try {
    ARG_CHECK(ctx && accum_dev, "ctx/accum_dev is NULL");
    ARG_CHECK(width > 0 && height > 0, "width/height must be positive");
    ARG_CHECK(out_rgb_dev || out_rgb8_dev, "no output buffer");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::launch_tonemap(static_cast<const float4*>(accum_dev), width, height, static_cast<float*>(out_rgb_dev),
                        static_cast<uint8_t*>(out_rgb8_dev), ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
} RT_API_CATCH

rt_status rt_selftest_rz(rt_context* ctx, const float* x, const float* y, size_t n, float* out) try {
    ARG_CHECK(ctx && (n == 0 || (x && y && out)), "ctx/x/y/out is NULL");
    if (n == 0) return RT_OK;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::PoolBuffer<float> dx, dy, dout;
    CUDA_TRY(dx.alloc(n, ctx->stream));
    cudaError_t e = dy.alloc(n, ctx->stream);
    if (e == cudaSuccess) e = dout.alloc(4 * n, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dx.get(), x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dy.get(), y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::launch_selftest_rz(dx.get(), dy.get(), n, dout.get(), ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout.get(), 4 * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("rt_selftest_rz: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    return RT_OK;
} RT_API_CATCH

rt_status rt_reduce_tonemap_peers(rt_context* ctx, const void* const* peer_accum_dev, int32_t n_peers, const void* multicast_accum,
                                  int32_t width, int32_t height, int32_t row_begin, int32_t row_end, void* out_rgb_dev,
                                  void* out_rgb8_dev, void* out_sum_dev) try {
    ARG_CHECK(ctx != nullptr, "ctx is NULL");
    ARG_CHECK(width > 0 && height > 0, "width/height must be positive");
    ARG_CHECK(row_begin >= 0 && row_begin <= row_end && row_end <= height, "bad row range");
    ARG_CHECK(n_peers >= 1 && n_peers <= 16, "n_peers must be in [1, 16]");
    ARG_CHECK(multicast_accum || peer_accum_dev, "no accumulator pointers");
    ARG_CHECK(out_rgb_dev || out_rgb8_dev || out_sum_dev, "no output buffer");
    if (peer_accum_dev)
        for (int k = 0; k < n_peers; ++k) ARG_CHECK(peer_accum_dev[k] != nullptr, "peer accumulator pointer is NULL");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::launch_reduce_tonemap(peer_accum_dev, n_peers, multicast_accum, width, height, row_begin, row_end,
                               static_cast<float*>(out_rgb_dev), static_cast<uint8_t*>(out_rgb8_dev),
                               static_cast<float4*>(out_sum_dev), ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
} RT_API_CATCH

rt_status rt_render(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, float* out_rgb, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_rgb, "ctx/scene/out_rgb is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    if ((st = grow(ctx->out_rgb, ctx->out_rgb_n, npix * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_rp(ctx, scene, to_device_params(*p), p->pipeline, ctx->accum, &local)) != RT_OK) return st;
    local.launches += 1;
    return finish_to_host(ctx, [&] { return tonemap_frames(ctx, p, 1); }, {ctx->out_rgb, out_rgb, npix * 3 * sizeof(float)}, local,
                          stats);
} RT_API_CATCH

size_t rt_jpeg_max_bytes(int32_t width, int32_t height) {
    if (width <= 0 || height <= 0) return 0;
    return rtd::jpeg_max_bytes(width, height);
}

rt_status rt_jpeg_encode_device(rt_context* ctx, const void* rgb8_dev, int32_t width, int32_t height, int32_t quality,
                                uint8_t* out_jpg, size_t cap, size_t* n_bytes, float* ms_device) try {
    ARG_CHECK(ctx && rgb8_dev && n_bytes, "ctx/rgb8_dev/n_bytes is NULL");
    ARG_CHECK(width > 0 && height > 0 && width < 65536 && height < 65536, "JPEG dimensions must be in [1, 65535]");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    return jpeg_from_device(ctx, static_cast<const uint8_t*>(rgb8_dev), width, height, quality, out_jpg, cap, n_bytes, ms_device);
} RT_API_CATCH

rt_status rt_jpeg_encode(rt_context* ctx, const uint8_t* rgb8, int32_t width, int32_t height, int32_t quality, uint8_t* out_jpg,
                         size_t cap, size_t* n_bytes) try {
    ARG_CHECK(ctx && rgb8 && n_bytes, "ctx/rgb8/n_bytes is NULL");
    ARG_CHECK(width > 0 && height > 0 && width < 65536 && height < 65536, "JPEG dimensions must be in [1, 65535]");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    const size_t npix = size_t(width) * size_t(height);
    if ((st = grow(ctx->rgb8, ctx->rgb8_n, npix * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemcpyAsync(ctx->rgb8, rgb8, npix * 3, cudaMemcpyHostToDevice, ctx->stream));
    return jpeg_from_device(ctx, ctx->rgb8, width, height, quality, out_jpg, cap, n_bytes, nullptr);
} RT_API_CATCH

rt_status rt_write_jpg(rt_context* ctx, const char* path, int32_t width, int32_t height, const uint8_t* rgb8, int32_t quality) try {
    ARG_CHECK(path != nullptr, "path is NULL");
    const size_t cap = rt_jpeg_max_bytes(width, height);
    std::vector<uint8_t> buf(cap);
    size_t n = 0;
    rt_status st = rt_jpeg_encode(ctx, rgb8, width, height, quality, buf.data(), cap, &n);
    if (st != RT_OK) return st;
    FILE* f = fopen(path, "wb");
    if (!f) {
        set_error("cannot open %s for writing", path);
        return RT_ERR_IO;
    }
    const bool ok = fwrite(buf.data(), 1, n, f) == n;
    fclose(f);
    if (!ok) {
        set_error("short write to %s", path);
        return RT_ERR_IO;
    }
    return RT_OK;
} RT_API_CATCH

rt_status rt_render_jpeg(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t quality, uint8_t* out_jpg,
                         size_t cap, size_t* n_bytes, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_jpg && n_bytes, "ctx/scene/out_jpg/n_bytes is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    ARG_CHECK(p->width < 65536 && p->height < 65536, "JPEG dimensions must be in [1, 65535]");
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    if ((st = grow(ctx->rgb8, ctx->rgb8_n, npix * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_rp(ctx, scene, to_device_params(*p), p->pipeline, ctx->accum, &local)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    rtd::launch_tonemap(ctx->accum, p->width, p->height, nullptr, ctx->rgb8, ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    float ms_jpg = 0.f;
    if ((st = jpeg_from_device(ctx, ctx->rgb8, p->width, p->height, quality, out_jpg, cap, n_bytes, &ms_jpg)) != RT_OK) return st;
    CUDA_TRY(cudaEventElapsedTime(&local.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    local.ms_d2h = ms_jpg; // device time of the JPEG passes; the D2H copy moves the finished file only
    local.launches += 8;
    if (stats) *stats = local;
    return RT_OK;
} RT_API_CATCH

rt_status rt_render_progressive(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t passes, float* out_rgb,
                                rt_progress_fn on_pass, void* user, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_rgb, "ctx/scene/out_rgb is NULL");
    ARG_CHECK(passes >= 1, "passes must be >= 1");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    if ((st = grow(ctx->out_rgb, ctx->out_rgb_n, npix * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats total;
    memset(&total, 0, sizeof total);
    for (int32_t k = 0; k < passes; ++k) {
        rt_render_params pk = *p;
        pk.sample_offset = p->sample_offset + k * p->spp; // Philox keys use the global sample index: no sample repeats
        rt_stats local;
        if ((st = render_rp(ctx, scene, to_device_params(pk), pk.pipeline, ctx->accum, &local)) != RT_OK) return st;
        // the accumulator carries the sample count per pixel, so the same finalisation works after every pass
        if ((st = tonemap_frames(ctx, p, 1)) != RT_OK) return st;
        CUDA_TRY(cudaMemcpyAsync(out_rgb, ctx->out_rgb, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        total.paths += local.paths;
        total.rays += local.rays;
        total.ms_total += local.ms_total;
        total.launches += local.launches + 1;
        total.iterations += local.iterations;
        if (on_pass && on_pass(k, (k + 1) * p->spp, out_rgb, user) != 0) break; // the caller asked to stop
    }
    if (stats) *stats = total;
    return RT_OK;
} RT_API_CATCH

void rt_default_denoise_params(rt_denoise_params* d) {
    if (!d) return;
    d->iterations = 3;
    d->feature_spp = 4;
    // the best worst case over C1 / C2 / C3 at 4 spp of a sweep of 216 settings (profiles/r03_denoise.md)
    d->sigma_color = 0.5f;
    d->sigma_normal = 1.0f;
    d->sigma_depth = 0.3f;
    d->sigma_albedo = 1.0f;
}

} // extern "C"

namespace {

rt_status check_denoise(const rt_denoise_params* d) {
    ARG_CHECK(d != nullptr, "denoise params is NULL");
    ARG_CHECK(d->iterations >= 0 && d->iterations <= 8, "iterations must be in [0, 8]");
    ARG_CHECK(d->feature_spp >= 1, "feature_spp must be >= 1");
    for (float s : {d->sigma_color, d->sigma_normal, d->sigma_depth, d->sigma_albedo})
        ARG_CHECK(std::isfinite(s) && s > 0.f, "sigmas must be positive and finite");
    return RT_OK;
}

rt_status features_into(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t feature_spp, float4* features) {
    rtd::DRenderParams rp = to_device_params(*p);
    rp.flags = 0; // the features describe the first hit of the reference estimator: no shadow rays
    rtd::launch_features(scene->d, rp, scene->d.nodes != nullptr, feature_spp, features, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

// d->iterations levels ping-ponging between two scratch planes, then the pixel finalisation of the last one
rt_status denoise_into(rt_context* ctx, const float4* accum, const float4* features, int32_t width, int32_t height,
                       const rt_denoise_params* d, float* out_rgb, uint8_t* out_rgb8) {
    if (d->iterations == 0) {
        rtd::launch_tonemap(accum, width, height, out_rgb, out_rgb8, ctx->sm_count, ctx->stream);
        CUDA_TRY(cudaGetLastError());
        return RT_OK;
    }
    const size_t npix = size_t(width) * size_t(height);
    rtd::PoolBuffer<float4> scratch;
    CUDA_TRY(scratch.alloc(2 * npix, ctx->stream));
    const float4* in = accum;
    float4* out = scratch.get();
    for (int32_t level = 0; level < d->iterations; ++level) {
        rtd::launch_atrous(in, level == 0, features, width, height, level, d->sigma_color, d->sigma_normal, d->sigma_depth,
                           d->sigma_albedo, out, ctx->stream);
        in = out;
        out = out == scratch.get() ? scratch.get() + npix : scratch.get();
    }
    rtd::launch_tonemap(in, width, height, out_rgb, out_rgb8, ctx->sm_count, ctx->stream);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("denoise: %s", cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    return RT_OK;
}

} // namespace

extern "C" {

rt_status rt_render_features_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t feature_spp,
                                    void* features_dev) try {
    ARG_CHECK(ctx && scene && features_dev, "ctx/scene/features_dev is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    ARG_CHECK(feature_spp >= 1, "feature_spp must be >= 1");
    ARG_CHECK(int64_t(p->sample_offset) + feature_spp <= INT32_MAX, "sample indices exceed 2^31");
    if ((st = make_current(ctx)) != RT_OK) return st;
    return features_into(ctx, scene, p, feature_spp, static_cast<float4*>(features_dev));
} RT_API_CATCH

rt_status rt_denoise_device(rt_context* ctx, const void* accum_dev, const void* features_dev, int32_t width, int32_t height,
                            const rt_denoise_params* d, void* out_rgb_dev, void* out_rgb8_dev) try {
    ARG_CHECK(ctx && accum_dev && features_dev, "ctx/accum_dev/features_dev is NULL");
    ARG_CHECK(width > 0 && height > 0, "width/height must be positive");
    ARG_CHECK(uint64_t(width) * uint64_t(height) < (1ull << 31), "frame has more than 2^31 pixels");
    ARG_CHECK(out_rgb_dev || out_rgb8_dev, "no output buffer");
    rt_status st = check_denoise(d);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    return denoise_into(ctx, static_cast<const float4*>(accum_dev), static_cast<const float4*>(features_dev), width, height, d,
                        static_cast<float*>(out_rgb_dev), static_cast<uint8_t*>(out_rgb8_dev));
} RT_API_CATCH

rt_status rt_render_denoised(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_denoise_params* d,
                             float* out_rgb, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_rgb, "ctx/scene/out_rgb is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = check_denoise(d)) != RT_OK) return st;
    ARG_CHECK(int64_t(p->sample_offset) + d->feature_spp <= INT32_MAX, "sample indices exceed 2^31");
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    if ((st = grow(ctx->out_rgb, ctx->out_rgb_n, npix * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_rp(ctx, scene, to_device_params(*p), p->pipeline, ctx->accum, &local)) != RT_OK) return st;
    rtd::PoolBuffer<float4> features;
    CUDA_TRY(features.alloc(2 * npix, ctx->stream));
    auto finalise = [&] {
        const rt_status s = features_into(ctx, scene, p, d->feature_spp, features.get());
        return s != RT_OK ? s : denoise_into(ctx, ctx->accum, features.get(), p->width, p->height, d, ctx->out_rgb, nullptr);
    };
    local.launches += 2 + uint32_t(d->iterations); // features, the levels, the finalisation
    return finish_to_host(ctx, finalise, {ctx->out_rgb, out_rgb, npix * 3 * sizeof(float)}, local, stats);
} RT_API_CATCH

void rt_default_adaptive_params(rt_adaptive_params* a) {
    if (!a) return;
    // the best worst case over C1 / C2 / C3 of a 36-setting sweep at equal budget, up to 0.03 dB (profiles/r04_adaptive.md)
    a->min_spp = 32;
    a->step_spp = 32;
    a->max_spp = 256;
    a->threshold = 1.f / 255.f;
}

} // extern "C"

namespace {

rt_status check_adaptive(const rt_render_params* p, const rt_adaptive_params* a) {
    ARG_CHECK(a != nullptr, "adaptive params is NULL");
    ARG_CHECK(a->min_spp >= 2 && a->min_spp % 2 == 0, "min_spp must be even and >= 2");
    ARG_CHECK(a->step_spp >= 2 && a->step_spp % 2 == 0, "step_spp must be even and >= 2");
    ARG_CHECK(a->max_spp >= a->min_spp && (a->max_spp - a->min_spp) % a->step_spp == 0, "max_spp must be min_spp + k * step_spp, k >= 0");
    ARG_CHECK(a->max_spp <= (1 << 24), "max_spp exceeds 2^24, up to which the float sample count is exact");
    ARG_CHECK(std::isfinite(a->threshold) && a->threshold >= 0.f, "threshold must be finite and >= 0");
    ARG_CHECK(int64_t(p->sample_offset) + a->max_spp <= INT32_MAX, "sample indices exceed 2^31");
    return RT_OK;
}

// The adaptive render (rt_adaptive.cu): pass 0 gives every pixel min_spp samples, every later pass step_spp samples to the
// pixels the selection kept; then accum = A + B (written) and, if error_dev, the final windowed error map.  Stream-ordered
// on the context stream, with one 4-byte read-back of the list length per pass.
rt_status adaptive_into(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_adaptive_params* a, float4* accum,
                        float* error_dev, int32_t* passes_out, rt_stats* stats) {
    cudaStream_t stream = ctx->stream;
    const uint32_t npix = uint32_t(p->width) * uint32_t(p->height);
    auto align = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t b_planes = align(2 * size_t(npix) * sizeof(float4)), b_px = align(size_t(npix) * sizeof(uint32_t));
    const size_t b_words = align(rtd::adapt_select_scratch_words(npix) * sizeof(uint32_t));
    rtd::PoolBuffer<char> mem; // planes A and B, the error map, two pixel lists, the selection's words, the list length
    CUDA_TRY(mem.alloc(b_planes + 3 * b_px + b_words + 256, stream));
    char* base = mem.get();
    float4* planes = reinterpret_cast<float4*>(base);
    float* e = reinterpret_cast<float*>(base + b_planes);
    uint32_t* list[2] = {reinterpret_cast<uint32_t*>(base + b_planes + b_px), reinterpret_cast<uint32_t*>(base + b_planes + 2 * b_px)};
    uint32_t* words = reinterpret_cast<uint32_t*>(base + b_planes + 3 * b_px);
    uint32_t* n_dev = reinterpret_cast<uint32_t*>(base + b_planes + 3 * b_px + b_words);
    CUDA_TRY(cudaMemsetAsync(planes, 0, 2 * size_t(npix) * sizeof(float4), stream));
    rt_status st = stats_begin(ctx, stats);
    if (st != RT_OK) return st;
    rtd::launch_adapt_iota(list[0], npix, stream);
    rtd::DRenderParams rp = to_device_params(*p);
    rp.adapt_first = uint32_t(p->sample_offset);
    rp.adapt_plane = npix;
    uint32_t n = npix, launches = 2, iterations = 0; // (iota and merge)
    int32_t done = 0, passes = 0, cur = 0;          // samples of every listed pixel so far, passes run, current list
    uint64_t paths = 0;
    for (;;) {
        rp.spp = passes == 0 ? a->min_spp : a->step_spp;
        rp.sample_offset = p->sample_offset + done;
        rp.adapt_pixels = list[cur];
        rp.div_npix = rtd::make_fastdiv(n);
        uint32_t l = 0, it = 0;
        if ((st = render_pass(ctx, scene, rp, p->pipeline, planes, &l, &it)) != RT_OK) return st;
        launches += l;
        iterations += it;
        paths += uint64_t(n) * uint64_t(rp.spp);
        done += rp.spp;
        ++passes;
        if (done >= a->max_spp) break;
        CUDA_TRY(rtd::launch_adapt_select(planes, p->width, p->height, list[cur], n, a->threshold, a->max_spp, e, words, list[cur ^ 1],
                                          n_dev, &l, stream));
        launches += l;
        uint32_t n_next = 0;
        CUDA_TRY(cudaMemcpyAsync(&n_next, n_dev, sizeof n_next, cudaMemcpyDeviceToHost, stream));
        CUDA_TRY(cudaStreamSynchronize(stream));
        if (n_next == 0) break;
        n = n_next;
        cur ^= 1;
    }
    rtd::launch_adapt_merge(planes, npix, accum, stream);
    if (error_dev) {
        rtd::launch_adapt_error_map(planes, p->width, p->height, e, error_dev, stream);
        launches += 2;
    }
    CUDA_TRY(cudaGetLastError());
    if (passes_out) *passes_out = passes;
    return stats_end(ctx, stats, paths, launches, iterations);
}

} // namespace

extern "C" {

rt_status rt_adaptive_error_device(rt_context* ctx, const void* planes_dev, int32_t width, int32_t height, void* error_dev) try {
    ARG_CHECK(ctx && planes_dev && error_dev, "ctx/planes_dev/error_dev is NULL");
    ARG_CHECK(width > 0 && height > 0, "width/height must be positive");
    ARG_CHECK(uint64_t(width) * uint64_t(height) < (1ull << 31), "frame has more than 2^31 pixels");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtd::PoolBuffer<float> e;
    CUDA_TRY(e.alloc(size_t(width) * size_t(height), ctx->stream));
    rtd::launch_adapt_error_map(static_cast<const float4*>(planes_dev), width, height, e.get(), static_cast<float*>(error_dev), ctx->stream);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) {
        set_error("adaptive error map: %s", cudaGetErrorString(err));
        return RT_ERR_CUDA;
    }
    return RT_OK;
} RT_API_CATCH

rt_status rt_render_adaptive_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_adaptive_params* a,
                                    void* accum_dev, void* error_dev, int32_t* passes, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && accum_dev, "ctx/scene/accum_dev is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = check_adaptive(p, a)) != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    return adaptive_into(ctx, scene, p, a, static_cast<float4*>(accum_dev), static_cast<float*>(error_dev), passes, stats);
} RT_API_CATCH

rt_status rt_render_adaptive(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_adaptive_params* a,
                             float* out_rgb, int32_t* out_spp, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_rgb, "ctx/scene/out_rgb is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = check_adaptive(p, a)) != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = grow(ctx->accum, ctx->accum_n, npix)) != RT_OK) return st;
    if ((st = grow(ctx->out_rgb, ctx->out_rgb_n, npix * 3)) != RT_OK) return st;
    rt_stats local;
    if ((st = adaptive_into(ctx, scene, p, a, ctx->accum, nullptr, nullptr, &local)) != RT_OK) return st;
    local.launches += 1;
    std::vector<float4> acc(out_spp ? npix : 0); // read back with the image, for the per-pixel sample counts
    st = finish_to_host(ctx, [&] { return tonemap_frames(ctx, p, 1); }, {ctx->out_rgb, out_rgb, npix * 3 * sizeof(float)}, local,
                        stats, {ctx->accum, acc.data(), acc.size() * sizeof(float4)});
    for (size_t i = 0; st == RT_OK && i < acc.size(); ++i) out_spp[i] = int32_t(acc[i].w); // (exact: counts stay below 2^24)
    return st;
} RT_API_CATCH

} // extern "C"

namespace {

rt_status check_frames(const rt_render_params* p, const rt_camera* cameras, int32_t n_frames) {
    ARG_CHECK(cameras != nullptr, "cameras is NULL");
    ARG_CHECK(n_frames >= 1, "n_frames must be >= 1");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    for (int32_t f = 0; f < n_frames; ++f) ARG_CHECK(rtd::camera_finite(cameras[f]), "camera parameter is not finite");
    ARG_CHECK(int64_t(p->sample_offset) + int64_t(n_frames) * int64_t(p->spp) <= INT32_MAX, "sample indices exceed 2^31 - 1");
    return RT_OK;
}

// A frame sequence as ONE render of n_frames * spp samples per pixel: sample block f (frame_of, rt_device.cuh) looks through
// cameras[f] and adds into accum + f * W * H, so the wavefront runs the frames back to back in one pool and one poll loop.
rt_status frames_into(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_camera* cameras, int32_t n_frames,
                      float4* accum, rt_stats* stats) {
    std::vector<rtd::DCamera> cams(static_cast<size_t>(n_frames));
    for (int32_t f = 0; f < n_frames; ++f) make_camera(cameras[f], cams[f]);
    rtd::PoolBuffer<rtd::DCamera> d_cams;
    CUDA_TRY(d_cams.alloc(cams.size(), ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(d_cams.get(), cams.data(), cams.size() * sizeof(rtd::DCamera), cudaMemcpyHostToDevice, ctx->stream));
    rtd::DRenderParams rp = to_device_params(*p);
    rp.spp = p->spp * n_frames; // <= 2^31 - 1: check_frames
    rp.frame_cams = d_cams.get();
    rp.div_spp = rtd::make_fastdiv(uint32_t(p->spp));
    return render_rp(ctx, scene, rp, p->pipeline, accum, stats);
}

} // namespace

extern "C" {

rt_status rt_render_frames_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_camera* cameras,
                                  int32_t n_frames, void* accum_dev, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && accum_dev, "ctx/scene/accum_dev is NULL");
    rt_status st = check_frames(p, cameras, n_frames);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    return frames_into(ctx, scene, p, cameras, n_frames, static_cast<float4*>(accum_dev), stats);
} RT_API_CATCH

rt_status rt_render_frames(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_camera* cameras,
                           int32_t n_frames, float* out_rgb, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_rgb, "ctx/scene/out_rgb is NULL");
    rt_status st = check_frames(p, cameras, n_frames);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height), total = npix * size_t(n_frames);
    if ((st = grow(ctx->accum, ctx->accum_n, total)) != RT_OK) return st;
    if ((st = grow(ctx->out_rgb, ctx->out_rgb_n, total * 3)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, total * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = frames_into(ctx, scene, p, cameras, n_frames, ctx->accum, &local)) != RT_OK) return st;
    local.launches += uint32_t(n_frames);
    return finish_to_host(ctx, [&] { return tonemap_frames(ctx, p, n_frames); }, {ctx->out_rgb, out_rgb, total * 3 * sizeof(float)},
                          local, stats);
} RT_API_CATCH

namespace {
struct OwnedCoefficients { // rt_jpeg_coefficients that owns its planes; `pub` must stay the first member
    rt_jpeg_coefficients pub;
    rtj::CoefficientImage img;
};
} // namespace

rt_status rt_jpeg_parse(const uint8_t* file, size_t n_bytes, rt_jpeg_coefficients** out) try {
    ARG_CHECK(file && out, "file/out is NULL");
    *out = nullptr;
    OwnedCoefficients* oc = new (std::nothrow) OwnedCoefficients();
    if (!oc) return RT_ERR_OOM;
    if (!rtj::decode_coefficients(file, n_bytes, oc->img)) {
        set_error("JPEG: %s", oc->img.error.c_str());
        delete oc;
        return RT_ERR_INVALID_ARG;
    }
    rt_jpeg_coefficients& p = oc->pub;
    memset(&p, 0, sizeof p);
    p.width = oc->img.width;
    p.height = oc->img.height;
    p.n_comp = oc->img.n_comp;
    p.h_max = oc->img.h_max;
    p.v_max = oc->img.v_max;
    p.progressive = oc->img.progressive ? 1 : 0;
    p.is_rgb = oc->img.is_rgb ? 1 : 0;
    for (int k = 0; k < oc->img.n_comp; ++k) {
        const rtj::Component& c = oc->img.comp[k];
        p.comp[k] = rt_jpeg_component{c.h, c.v, c.tq, c.x, c.y, c.w2, c.h2, c.blocks_w, c.blocks_h, c.coeff.data()};
    }
    memcpy(p.dequant, oc->img.dequant, sizeof p.dequant);
    *out = &oc->pub;
    return RT_OK;
} RT_API_CATCH

void rt_jpeg_coefficients_free(rt_jpeg_coefficients* c) {
    if (c) delete reinterpret_cast<OwnedCoefficients*>(c);
}

rt_status rt_jpeg_decode(rt_context* ctx, const uint8_t* file, size_t n_bytes, float** out_pixels, int32_t* width, int32_t* height,
                         int32_t* channels, float* ms_device) try {
    ARG_CHECK(ctx && file && out_pixels && width && height && channels, "ctx/file/out pointers are NULL");
    *out_pixels = nullptr;
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    rtj::CoefficientImage img;
    if (!rtj::decode_coefficients(file, n_bytes, img)) {
        set_error("JPEG: %s", img.error.c_str());
        return RT_ERR_INVALID_ARG;
    }
    const int ch = img.n_comp == 1 ? 1 : 3;
    const size_t n = size_t(img.width) * size_t(img.height) * size_t(ch);
    rtd::PoolBuffer<float> d_out;
    CUDA_TRY(d_out.alloc(n, ctx->stream));
    cudaError_t e = rtd::jpeg_pixels_device(img, d_out.get(), ctx->stream, ms_device);
    float* host = e == cudaSuccess ? static_cast<float*>(malloc(n * sizeof(float))) : nullptr;
    if (e == cudaSuccess && host) {
        e = cudaMemcpyAsync(host, d_out.get(), n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    if (e != cudaSuccess) {
        free(host);
        set_error("jpeg_decode: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return RT_ERR_CUDA;
    }
    if (!host) return RT_ERR_OOM;
    *out_pixels = host;
    *width = img.width;
    *height = img.height;
    *channels = ch;
    return RT_OK;
} RT_API_CATCH

rt_status rt_image_load(rt_context* ctx, const char* path, float** out_rgb, int32_t* width, int32_t* height) try {
    ARG_CHECK(path && out_rgb && width && height, "path/out pointers are NULL");
    *out_rgb = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) {
        set_error("cannot open %s", path);
        return RT_ERR_IO;
    }
    std::vector<uint8_t> bytes;
    uint8_t buf[65536];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) bytes.insert(bytes.end(), buf, buf + n);
    fclose(f);
    if (bytes.size() >= 2 && bytes[0] == 'P' && (bytes[1] == '6' || bytes[1] == '5')) return rt_read_ppm_f32(path, out_rgb, width, height);
    ARG_CHECK(ctx != nullptr, "a JPEG file needs a context (the pixel stages run on the device)");
    float* px = nullptr;
    int32_t ch = 0;
    rt_status st = rt_jpeg_decode(ctx, bytes.data(), bytes.size(), &px, width, height, &ch, nullptr);
    if (st != RT_OK) return st;
    if (ch == 3) {
        *out_rgb = px;
        return RT_OK;
    }
    float* rgb = static_cast<float*>(malloc(size_t(*width) * size_t(*height) * 3 * sizeof(float)));
    if (!rgb) {
        free(px);
        return RT_ERR_OOM;
    }
    st = rt_image_to_rgb(px, *width, *height, ch, rgb);
    free(px);
    if (st != RT_OK) {
        free(rgb);
        return st;
    }
    *out_rgb = rgb;
    return RT_OK;
} RT_API_CATCH

} // extern "C"
