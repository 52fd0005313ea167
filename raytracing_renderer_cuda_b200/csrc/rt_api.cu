// rt_api.cu — C-ABI of librt_b200.so (include/rt_api.h): context, scene upload +
// acceleration-structure build, render / accumulate / tonemap entry points.
// Host logic only; the kernels live in rt_kernels.cu / rt_wavefront.cu / rt_lbvh.cu.
#include <algorithm>
#include <cfenv>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <string>
#include <vector>

#include "rt_bvh_host.hpp"
#include "rt_jpeg.cuh"
#include "rt_jpeg_decode.cuh"
#include "rt_kernels.cuh"
#include "rt_lbvh.cuh"

namespace {

thread_local std::string g_last_error;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

} // namespace
namespace rtd {
namespace {
thread_local cudaMemPool_t g_thread_pool = nullptr;
}
void set_thread_mempool(cudaMemPool_t pool) { g_thread_pool = pool; }
cudaError_t malloc_async_bytes(void** p, size_t bytes, cudaStream_t st) {
    return g_thread_pool ? cudaMallocFromPoolAsync(p, bytes, g_thread_pool, st) : cudaMallocAsync(p, bytes, st);
}
// message hook for the host-only translation unit (rt_host.cpp), which has no CUDA error paths of its own
void set_error_message(const char* msg) { g_last_error = msg ? msg : ""; }
} // namespace rtd
namespace {

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (expr);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__));   \
            return e__ == cudaErrorMemoryAllocation ? RT_ERR_OOM : RT_ERR_CUDA;                 \
        }                                                                                       \
    } while (0)

// Every rt_status entry point is a function-try-block closed by this: nothing propagates through the C ABI
// (SURVEY.md 8b "no exceptions across the boundary"); host containers that cannot grow are RT_ERR_OOM.
#define RT_API_CATCH                                   \
    catch (const std::bad_alloc&) {                    \
        set_error("out of host memory");               \
        return RT_ERR_OOM;                             \
    }                                                  \
    catch (const std::exception& e) {                  \
        set_error("unexpected exception: %s", e.what()); \
        return RT_ERR_INVALID_ARG;                     \
    }
#define ARG_CHECK(cond, msg)                  \
    do {                                      \
        if (!(cond)) {                        \
            set_error("invalid argument: %s", msg); \
            return RT_ERR_INVALID_ARG;        \
        }                                     \
    } while (0)

} // namespace

#include "rt_internal.hpp"

namespace {

rt_status make_current(const rt_context* ctx) {
    CUDA_TRY(cudaSetDevice(ctx->device));
    rtd::set_thread_mempool(ctx->pool);
    return RT_OK;
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

} // namespace
namespace rtd {
// every parameter of a camera finite (scene descriptions, frame sequences, rt_orbit_cameras)
bool camera_finite(const rt_camera& c) {
    auto finite3 = [](const float* v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); };
    return finite3(c.lookfrom) && finite3(c.lookat) && finite3(c.up) && std::isfinite(c.vfov) && std::isfinite(c.aspect) &&
           std::isfinite(c.aperture) && std::isfinite(c.focus_dist) && std::isfinite(c.time0) && std::isfinite(c.time1);
}
} // namespace rtd
namespace {

// camera ctor (camera.h:7-31) in host float arithmetic
void make_camera(const rt_camera& c, rtd::DCamera& out) {
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
    for (uint32_t i = 0; i < d->n_materials; ++i) {
        const rt_material& m = d->materials[i];
        ARG_CHECK(m.kind <= RT_MAT_EMITTER, "bad material kind");
        if (m.kind == RT_MAT_LAMBERTIAN || m.kind == RT_MAT_EMITTER)
            ARG_CHECK(m.texture >= 0 && uint32_t(m.texture) < d->n_textures, "material texture out of range");
    }
    // non-finite geometry would reach the builders' bin arithmetic (undefined for NaN / infinity) and the slab tests
    auto finite3 = [](const float* v) { return std::isfinite(v[0]) && std::isfinite(v[1]) && std::isfinite(v[2]); };
    for (uint32_t i = 0; i < d->n_spheres; ++i) {
        const rt_sphere& sp = d->spheres[i];
        ARG_CHECK(sp.material < d->n_materials, "sphere material out of range");
        ARG_CHECK(finite3(sp.center0) && finite3(sp.center1) && std::isfinite(sp.radius) && std::isfinite(sp.time0) &&
                      std::isfinite(sp.time1),
                  "sphere centre / radius / time is not finite");
    }
    ARG_CHECK(rtd::camera_finite(d->camera), "camera parameter is not finite");
    return RT_OK;
}

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

rt_status ensure_accum(rt_context* ctx, size_t npix) {
    if (ctx->accum_px < npix) {
        if (ctx->accum) cudaFree(ctx->accum);
        ctx->accum = nullptr;
        ctx->accum_px = 0;
        CUDA_TRY(cudaMalloc(&ctx->accum, npix * sizeof(float4)));
        ctx->accum_px = npix;
    }
    return RT_OK;
}

rt_status ensure_out(rt_context* ctx, size_t npix) {
    if (ctx->out_px < npix) {
        if (ctx->out_rgb) cudaFree(ctx->out_rgb);
        ctx->out_rgb = nullptr;
        ctx->out_px = 0;
        CUDA_TRY(cudaMalloc(&ctx->out_rgb, npix * 3 * sizeof(float)));
        ctx->out_px = npix;
    }
    return RT_OK;
}

rt_status ensure_rgb8(rt_context* ctx, size_t npix) {
    if (ctx->rgb8_px < npix) {
        if (ctx->rgb8) cudaFree(ctx->rgb8);
        ctx->rgb8 = nullptr;
        ctx->rgb8_px = 0;
        CUDA_TRY(cudaMalloc(&ctx->rgb8, npix * 3));
        ctx->rgb8_px = npix;
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

// Core: adds rp.spp samples per pixel into accum (device).  Fills stats if requested
// (which synchronises the stream).
rt_status render_rp(rt_context* ctx, const rt_scene* scene, const rtd::DRenderParams& rp, uint32_t pipeline, float4* accum,
                    rt_stats* stats) {
    uint32_t launches = 0, iterations = 0;
    if (stats) {
        CUDA_TRY(cudaMemsetAsync(ctx->d_ray_counter, 0, sizeof(unsigned long long), ctx->stream));
        CUDA_TRY(cudaEventRecord(ctx->ev[0], ctx->stream));
    }
    rt_status st = render_pass(ctx, scene, rp, pipeline, accum, &launches, &iterations);
    if (st != RT_OK) return st;
    if (stats) {
        CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
        unsigned long long rays = 0;
        CUDA_TRY(cudaMemcpyAsync(&rays, ctx->d_ray_counter, sizeof rays, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        memset(stats, 0, sizeof *stats);
        CUDA_TRY(cudaEventElapsedTime(&stats->ms_total, ctx->ev[0], ctx->ev[1]));
        stats->paths = uint64_t(rp.width) * uint64_t(rp.height) * uint64_t(rp.spp);
        stats->rays = rays;
        stats->launches = launches;
        stats->iterations = iterations;
    }
    return RT_OK;
}

rt_status render_into(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, float4* accum, rt_stats* stats) {
    return render_rp(ctx, scene, to_device_params(*p), p->pipeline, accum, stats);
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

rt_status rt_scene_create(rt_context* ctx, const rt_scene_desc* desc, rt_scene** out) try {
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

    // ---- primitives: static spheres first (stable), SoA float4 arrays ----
    std::vector<uint32_t> order;
    order.reserve(n);
    for (uint32_t i = 0; i < n; ++i)
        if (!(desc->spheres[i].flags & RT_SPHERE_MOVING)) order.push_back(i);
    const uint32_t n_static = uint32_t(order.size());
    for (uint32_t i = 0; i < n; ++i)
        if (desc->spheres[i].flags & RT_SPHERE_MOVING) order.push_back(i);

    // ---- acceleration structure: which one ----
    uint32_t mode = desc->bvh_mode;
    if (mode == RT_BVH_AUTO) mode = n <= 12 ? RT_BVH_NONE : (n <= 200000 ? RT_BVH_HOST_SAH : RT_BVH_GPU_LBVH);
    if (n < 2) mode = RT_BVH_NONE;

    std::vector<float4> ha(n), hb(n);
    std::vector<uint4> hc(n);
    std::vector<rth::Box> boxes(mode == RT_BVH_HOST_SAH ? n : 0);
    {
        // c1 - c0 rounded toward zero (== __fsub_rz, vec3 operator- of moving_sphere::center, sphere.h:51).  The rounding
        // mode is switched once around this loop, not per operation: at 10^6 spheres a per-call switch
        // cost 150 ms of every scene upload.
        const int old_round = std::fegetround();
        std::fesetround(FE_TOWARDZERO);
        for (uint32_t k = 0; k < n; ++k) {
            const rt_sphere& sp = desc->spheres[order[k]];
            volatile float dx = sp.center1[0], dy = sp.center1[1], dz = sp.center1[2];
            dx = dx - sp.center0[0];
            dy = dy - sp.center0[1];
            dz = dz - sp.center0[2];
            hb[k] = make_float4(dx, dy, dz, sp.time0);
        }
        std::fesetround(old_round);
    }
    for (uint32_t k = 0; k < n; ++k) {
        const rt_sphere& sp = desc->spheres[order[k]];
        ha[k] = make_float4(sp.center0[0], sp.center0[1], sp.center0[2], sp.radius);
        float dt = sp.time1 - sp.time0; // FADD(RN) in the reference's SASS (sphere.h:51)
        uint32_t dt_bits;
        memcpy(&dt_bits, &dt, 4);
        hc[k] = make_uint4(dt_bits, sp.material, sp.id, order[k]);
        const bool moving = (sp.flags & RT_SPHERE_MOVING) != 0;
        if (mode == RT_BVH_HOST_SAH) boxes[k] = rth::sphere_box(sp.center0, moving ? sp.center1 : sp.center0, sp.radius);
    }

    std::vector<rth::NodeHost> nodes;
    rth::BvhStats bstats;
    const auto t_build0 = std::chrono::steady_clock::now();
    if (mode == RT_BVH_HOST_SAH) rth::build_bvh_sah(boxes, nodes, &bstats);
    const auto t_build1 = std::chrono::steady_clock::now();

    // ---- upload ----
    float4 *da = nullptr, *db = nullptr;
    uint4* dc = nullptr;
    rtd::BvhNode* dnodes = nullptr;
    rtd::DMaterial* dmats = nullptr;
    rtd::DTexture* dtexs = nullptr;
    if ((st = dev_alloc(s, &da, n)) != RT_OK) return st;
    if ((st = dev_alloc(s, &db, n)) != RT_OK) return st;
    if ((st = dev_alloc(s, &dc, n)) != RT_OK) return st;
    cudaStream_t stream = ctx->stream;
    if (n) {
        CUDA_TRY(cudaMemcpyAsync(da, ha.data(), n * sizeof(float4), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(db, hb.data(), n * sizeof(float4), cudaMemcpyHostToDevice, stream));
        CUDA_TRY(cudaMemcpyAsync(dc, hc.data(), n * sizeof(uint4), cudaMemcpyHostToDevice, stream));
    }
    float lbvh_ms = 0.f;
    uint32_t bvh_root = 0;
    uint32_t n_nodes = 0;
    if (mode == RT_BVH_HOST_SAH) {
        n_nodes = uint32_t(nodes.size());
        if ((st = dev_alloc(s, &dnodes, n_nodes)) != RT_OK) return st;
        CUDA_TRY(cudaMemcpyAsync(dnodes, nodes.data(), n_nodes * sizeof(rtd::BvhNode), cudaMemcpyHostToDevice, stream));
    } else if (mode == RT_BVH_GPU_LBVH) {
        n_nodes = n - 1;
        if ((st = dev_alloc(s, &dnodes, n_nodes)) != RT_OK) return st;
        // Outsized primitives (the r = 1000 ground every scene of this renderer has) would sit deep in a Morton-ordered
        // tree and inflate the boxes of all their ancestors, so every ray would walk that whole chain.  They are kept
        // out of the LBVH and hung above its root instead: root -> (big_k, (... (big_0, LBVH root))).
        std::vector<uint32_t> big, normal;
        {
            std::vector<float> radii(n);
            for (uint32_t k = 0; k < n; ++k) radii[k] = std::fabs(ha[k].w);
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
        uint32_t* d_ids = nullptr;
        if (!big.empty()) {
            CUDA_TRY(rtd::malloc_async(&d_ids, m * sizeof(uint32_t), stream));
            CUDA_TRY(cudaMemcpyAsync(d_ids, normal.data(), m * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        }
        float rb[6];
        cudaError_t e = rtd::lbvh_build(da, db, n_static, d_ids, m, dnodes, stream, &lbvh_ms, &bstats.depth, rb);
        if (d_ids) cudaFreeAsync(d_ids, stream);
        if (e != cudaSuccess) {
            set_error("GPU LBVH build failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
        if (!big.empty()) {
            std::vector<rth::NodeHost> chain(big.size());
            rth::Box below{{rb[0], rb[1], rb[2]}, {rb[3], rb[4], rb[5]}};
            int32_t below_ref = 0; // the LBVH root
            for (size_t k = 0; k < big.size(); ++k) {
                const rt_sphere& sp = desc->spheres[order[big[k]]];
                const bool moving = (sp.flags & RT_SPHERE_MOVING) != 0;
                rth::Box bb = rth::sphere_box(sp.center0, moving ? sp.center1 : sp.center0, sp.radius);
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
            CUDA_TRY(cudaMemcpyAsync(dnodes + (m - 1), chain.data(), chain.size() * sizeof(rtd::BvhNode), cudaMemcpyHostToDevice, stream));
            CUDA_TRY(cudaStreamSynchronize(stream)); // `chain` is a pageable host buffer
            bvh_root = uint32_t(below_ref);
            bstats.depth += uint32_t(big.size());
        }
    }
    rtd::BvhNodeCH* dnodes_ch = nullptr;
    if (dnodes && n_nodes) { // the form the binary traversal reads
        if ((st = dev_alloc(s, &dnodes_ch, n_nodes)) != RT_OK) return st;
        cudaError_t e = rtd::bvh_nodes_ch(dnodes, n_nodes, dnodes_ch, stream);
        if (e != cudaSuccess) {
            set_error("BVH node conversion failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
    }
    rtd::BvhNode4* dnodes4 = nullptr;
    rtd::BvhNode4Q* dnodes4q = nullptr;
    uint32_t n_nodes4 = 0, root4 = 0;
    if (dnodes && n_nodes) { // the 4-wide form the persistent-lane kernel walks (half the dependent node fetches per ray)
        if ((st = dev_alloc(s, &dnodes4, n_nodes / 2 + 64)) != RT_OK) return st;
        rtd::BvhNode4* scratch = nullptr; // worst case (a degenerate chain) every binary node survives
        CUDA_TRY(rtd::malloc_async(&scratch, size_t(n_nodes) * sizeof(rtd::BvhNode4), stream));
        cudaError_t e = rtd::bvh_collapse4(dnodes, n_nodes, bvh_root, bstats.depth, scratch, &n_nodes4, &root4, stream);
        if (e == cudaSuccess && n_nodes4 <= n_nodes / 2 + 64) {
            e = cudaMemcpyAsync(dnodes4, scratch, size_t(n_nodes4) * sizeof(rtd::BvhNode4), cudaMemcpyDeviceToDevice, stream);
        } else if (e == cudaSuccess) { // unusually deep tree: keep the big array itself
            s->allocs.push_back(scratch);
            dnodes4 = scratch;
            scratch = nullptr;
        }
        if (scratch) cudaFreeAsync(scratch, stream);
        if (e != cudaSuccess) {
            set_error("4-wide BVH collapse failed: %s", cudaGetErrorString(e));
            return RT_ERR_CUDA;
        }
        // ... and the 64-byte quantised form of the same nodes (kept only when every node is representable)
        if (n_nodes4 && !getenv("RT_NO_BVH4Q")) {
            if ((st = dev_alloc(s, &dnodes4q, n_nodes4)) != RT_OK) return st;
            bool quant_ok = false;
            e = rtd::bvh_quantize4(dnodes4, n_nodes4, dnodes4q, &quant_ok, stream);
            if (e != cudaSuccess) {
                set_error("4-wide BVH quantisation failed: %s", cudaGetErrorString(e));
                return RT_ERR_CUDA;
            }
            if (!quant_ok) dnodes4q = nullptr; // (the memory stays with the scene; the walk uses the 128-byte nodes)
        }
    }
    if (bstats.depth > RT_BVH_STACK_DEPTH) {
        set_error("BVH depth %u exceeds the traversal stack (%d)", bstats.depth, RT_BVH_STACK_DEPTH);
        return RT_ERR_UNSUPPORTED;
    }

    std::vector<rtd::DMaterial> hm(desc->n_materials);
    for (uint32_t i = 0; i < desc->n_materials; ++i) {
        const rt_material& m = desc->materials[i];
        hm[i] = rtd::DMaterial{m.kind, m.texture, m.albedo[0], m.albedo[1], m.albedo[2], m.param, 0.f, 0.f};
    }
    std::vector<rtd::DTexture> ht(desc->n_textures);
    for (uint32_t i = 0; i < desc->n_textures; ++i) {
        const rt_texture& t = desc->textures[i];
        ht[i] = rtd::DTexture{t.kind,      t.even,      t.odd,       t.image,   t.color1[0], t.color1[1],
                              t.color1[2], t.density,   t.color2[0], t.color2[1], t.color2[2], t.hardness};
    }
    if ((st = dev_alloc(s, &dmats, hm.size())) != RT_OK) return st;
    if ((st = dev_alloc(s, &dtexs, ht.size())) != RT_OK) return st;
    if (!hm.empty()) CUDA_TRY(cudaMemcpyAsync(dmats, hm.data(), hm.size() * sizeof(rtd::DMaterial), cudaMemcpyHostToDevice, stream));
    if (!ht.empty()) CUDA_TRY(cudaMemcpyAsync(dtexs, ht.data(), ht.size() * sizeof(rtd::DTexture), cudaMemcpyHostToDevice, stream));

    // ---- image textures: float RGB -> float4 cudaArray + point-sampled texture object ----
    for (uint32_t i = 0; i < desc->n_images; ++i) {
        const rt_image& im = desc->images[i];
        const size_t texels = size_t(im.width) * size_t(im.height);
        float* d_rgb = nullptr;
        float4* d_rgba = nullptr;
        CUDA_TRY(rtd::malloc_async(&d_rgb, texels * 3 * sizeof(float), stream));
        cudaError_t e = rtd::malloc_async(&d_rgba, texels * sizeof(float4), stream);
        if (e != cudaSuccess) {
            cudaFreeAsync(d_rgb, stream);
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
        e = cudaMemcpyAsync(d_rgb, im.rgb, texels * 3 * sizeof(float), cudaMemcpyHostToDevice, stream);
        if (e == cudaSuccess) {
            rtd::launch_rgb_to_rgba(d_rgb, d_rgba, texels, ctx->sm_count, stream);
            if (!arr) e = cudaMallocArray(&arr, &cd, size_t(im.width), size_t(im.height));
        }
        if (e == cudaSuccess) {
            s->arrays.push_back(rt_context::CachedArray{im.width, im.height, arr});
            e = cudaMemcpy2DToArrayAsync(arr, 0, 0, d_rgba, size_t(im.width) * sizeof(float4), size_t(im.width) * sizeof(float4),
                                         size_t(im.height), cudaMemcpyDeviceToDevice, stream);
        }
        cudaFreeAsync(d_rgb, stream);
        cudaFreeAsync(d_rgba, stream);
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
        s->d.images[i] = rtd::DImage{tex, im.width, im.height};
        s->info.device_bytes += texels * sizeof(float4);
    }
    CUDA_TRY(cudaStreamSynchronize(stream));
    CUDA_TRY(cudaGetLastError());

    s->d.sph_a = da;
    s->d.sph_b = db;
    s->d.sph_c = dc;
    s->d.n_spheres = n;
    s->d.n_static = n_static;
    s->d.nodes = dnodes;
    s->d.nodes_ch = dnodes_ch;
    s->d.nodes4 = dnodes4;
    s->d.nodes4q = dnodes4q;
    s->d.n_nodes4 = n_nodes4;
    s->d.root4 = root4;
    s->d.n_nodes = n_nodes;
    s->d.root = bvh_root;
    s->d.mats = dmats;
    s->d.texs = dtexs;
    s->d.n_list = 0;
    if (mode == RT_BVH_NONE && n != 0 && n <= RT_LIST_MAX) { // the list in the constant bank (DScene::lst_*)
        s->d.n_list = n;
        for (uint32_t k = 0; k < n; ++k) {
            s->d.lst_a[k] = ha[k];
            s->d.lst_b[k] = hb[k];
            memcpy(&s->d.lst_dt[k], &hc[k].x, 4);
        }
    }
    s->d.has_noise = 0;
    for (const auto& t : ht)
        if (t.kind == RT_TEX_NOISE_PERLIN || t.kind == RT_TEX_NOISE_TURBULANCE || t.kind == RT_TEX_NOISE_MARBLE || t.kind == RT_TEX_WOOD) s->d.has_noise = 1;
    make_camera(desc->camera, s->d.cam);
    // emitter spheres for RT_RENDER_EMITTER_SAMPLING: device primitive indices in the caller's list order
    s->d.n_lights = 0;
    {
        std::vector<uint32_t> where(n); // list ordinal -> device index
        for (uint32_t k = 0; k < n; ++k) where[order[k]] = k;
        for (uint32_t i = 0; i < n && s->d.n_lights < RT_MAX_LIGHTS; ++i)
            if (desc->materials[desc->spheres[i].material].kind == RT_MAT_EMITTER) s->d.lights[s->d.n_lights++] = where[i];
        for (uint32_t k = s->d.n_lights; k < RT_MAX_LIGHTS; ++k) s->d.lights[k] = 0;
    }

    const auto t_end = std::chrono::steady_clock::now();
    s->info.n_spheres = n;
    s->info.n_nodes = n_nodes;
    s->info.bvh_mode = mode;
    s->info.bvh_depth = bstats.depth;
    s->info.sah_cost = bstats.sah_cost;
    s->info.ms_build = mode == RT_BVH_GPU_LBVH ? lbvh_ms
                                               : std::chrono::duration<float, std::milli>(t_build1 - t_build0).count();
    s->info.ms_upload = std::chrono::duration<float, std::milli>(t_end - t_begin).count() -
                        std::chrono::duration<float, std::milli>(t_build1 - t_build0).count();
    guard.s = nullptr;
    *out = s;
    return RT_OK;
} RT_API_CATCH

void rt_scene_destroy(rt_scene* scene) {
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

rt_status rt_scene_get_info(const rt_scene* scene, rt_scene_info* info) try {
    ARG_CHECK(scene && info, "scene/info is NULL");
    *info = scene->info;
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
    rt_ray* d_rays = nullptr;
    rt_hit* d_hits = nullptr;
    CUDA_TRY(rtd::malloc_async(&d_rays, n * sizeof(rt_ray), ctx->stream));
    cudaError_t e = rtd::malloc_async(&d_hits, n * sizeof(rt_hit), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::launch_trace_primary(scene->d, d_rays, n, tmin, use_bvh, d_hits, ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(hits, d_hits, n * sizeof(rt_hit), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(d_rays, ctx->stream);
    if (d_hits) cudaFreeAsync(d_hits, ctx->stream);
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
    rt_ray* d_rays = nullptr;
    rt_shade_sample* d_out = nullptr;
    CUDA_TRY(rtd::malloc_async(&d_rays, n * sizeof(rt_ray), ctx->stream));
    cudaError_t e = rtd::malloc_async(&d_out, n * sizeof(rt_shade_sample), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::DRenderParams rp = to_device_params(*p);
        rp.flags = 0; // the probe reports the reference estimator's terms (rt_shade_sample carries no path weight)
        rtd::launch_shade_probe(scene->d, rp, d_rays, n, use_bvh != 0, d_out, ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, n * sizeof(rt_shade_sample), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFreeAsync(d_rays, ctx->stream);
    if (d_out) cudaFreeAsync(d_out, ctx->stream);
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
    return render_into(ctx, scene, p, static_cast<float4*>(accum_dev), stats);
} RT_API_CATCH

rt_status rt_render_accum(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, float* out_accum, rt_stats* stats) try {
    ARG_CHECK(ctx && scene && out_accum, "ctx/scene/out_accum is NULL");
    rt_status st = check_params(p);
    if (st != RT_OK) return st;
    if ((st = make_current(ctx)) != RT_OK) return st;
    const size_t npix = size_t(p->width) * size_t(p->height);
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_into(ctx, scene, p, ctx->accum, &local)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_accum, ctx->accum, npix * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_d2h, ctx->ev[2], ctx->ev[3]));
    if (stats) *stats = local;
    return RT_OK;
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
    float *dx = nullptr, *dy = nullptr, *dout = nullptr;
    CUDA_TRY(rtd::malloc_async(&dx, n * sizeof(float), ctx->stream));
    cudaError_t e = rtd::malloc_async(&dy, n * sizeof(float), ctx->stream);
    if (e == cudaSuccess) e = rtd::malloc_async(&dout, 4 * n * sizeof(float), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dx, x, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dy, y, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        rtd::launch_selftest_rz(dx, dy, n, dout, ctx->stream);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, dout, 4 * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (dx) cudaFreeAsync(dx, ctx->stream);
    if (dy) cudaFreeAsync(dy, ctx->stream);
    if (dout) cudaFreeAsync(dout, ctx->stream);
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
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    if ((st = ensure_out(ctx, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_into(ctx, scene, p, ctx->accum, &local)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    rtd::launch_tonemap(ctx->accum, p->width, p->height, ctx->out_rgb, nullptr, ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_rgb, ctx->out_rgb, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_d2h, ctx->ev[2], ctx->ev[3]));
    local.launches += 1;
    if (stats) *stats = local;
    return RT_OK;
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
    if ((st = ensure_rgb8(ctx, npix)) != RT_OK) return st;
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
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    if ((st = ensure_rgb8(ctx, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_into(ctx, scene, p, ctx->accum, &local)) != RT_OK) return st;
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
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    if ((st = ensure_out(ctx, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats total;
    memset(&total, 0, sizeof total);
    for (int32_t k = 0; k < passes; ++k) {
        rt_render_params pk = *p;
        pk.sample_offset = p->sample_offset + k * p->spp; // Philox keys use the global sample index: no sample repeats
        rt_stats local;
        if ((st = render_into(ctx, scene, &pk, ctx->accum, &local)) != RT_OK) return st;
        // the accumulator carries the sample count per pixel, so the same finalisation works after every pass
        rtd::launch_tonemap(ctx->accum, p->width, p->height, ctx->out_rgb, nullptr, ctx->sm_count, ctx->stream);
        CUDA_TRY(cudaGetLastError());
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
    float4* scratch = nullptr;
    CUDA_TRY(rtd::malloc_async(&scratch, 2 * npix * sizeof(float4), ctx->stream));
    const float4* in = accum;
    float4* out = scratch;
    for (int32_t level = 0; level < d->iterations; ++level) {
        rtd::launch_atrous(in, level == 0, features, width, height, level, d->sigma_color, d->sigma_normal, d->sigma_depth,
                           d->sigma_albedo, out, ctx->stream);
        in = out;
        out = out == scratch ? scratch + npix : scratch;
    }
    rtd::launch_tonemap(in, width, height, out_rgb, out_rgb8, ctx->sm_count, ctx->stream);
    const cudaError_t e = cudaGetLastError();
    cudaFreeAsync(scratch, ctx->stream);
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
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    if ((st = ensure_out(ctx, npix)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, npix * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = render_into(ctx, scene, p, ctx->accum, &local)) != RT_OK) return st;
    float4* features = nullptr;
    CUDA_TRY(rtd::malloc_async(&features, 2 * npix * sizeof(float4), ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    st = features_into(ctx, scene, p, d->feature_spp, features);
    if (st == RT_OK) st = denoise_into(ctx, ctx->accum, features, p->width, p->height, d, ctx->out_rgb, nullptr);
    cudaFreeAsync(features, ctx->stream);
    if (st != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_rgb, ctx->out_rgb, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_d2h, ctx->ev[2], ctx->ev[3]));
    local.launches += 2 + uint32_t(d->iterations); // features, the levels, the finalisation
    if (stats) *stats = local;
    return RT_OK;
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
    char* base = nullptr; // planes A and B, the error map, two pixel lists, the selection's words, the list length
    CUDA_TRY(rtd::malloc_async(&base, b_planes + 3 * b_px + b_words + 256, stream));
    float4* planes = reinterpret_cast<float4*>(base);
    float* e = reinterpret_cast<float*>(base + b_planes);
    uint32_t* list[2] = {reinterpret_cast<uint32_t*>(base + b_planes + b_px), reinterpret_cast<uint32_t*>(base + b_planes + 2 * b_px)};
    uint32_t* words = reinterpret_cast<uint32_t*>(base + b_planes + 3 * b_px);
    uint32_t* n_dev = reinterpret_cast<uint32_t*>(base + b_planes + 3 * b_px + b_words);
    const rt_status st = [&]() -> rt_status {
        CUDA_TRY(cudaMemsetAsync(planes, 0, 2 * size_t(npix) * sizeof(float4), stream));
        CUDA_TRY(cudaMemsetAsync(ctx->d_ray_counter, 0, sizeof(unsigned long long), stream));
        CUDA_TRY(cudaEventRecord(ctx->ev[0], stream));
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
            const rt_status s = render_pass(ctx, scene, rp, p->pipeline, planes, &l, &it);
            if (s != RT_OK) return s;
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
        if (stats) {
            CUDA_TRY(cudaEventRecord(ctx->ev[1], stream));
            unsigned long long rays = 0;
            CUDA_TRY(cudaMemcpyAsync(&rays, ctx->d_ray_counter, sizeof rays, cudaMemcpyDeviceToHost, stream));
            CUDA_TRY(cudaStreamSynchronize(stream));
            memset(stats, 0, sizeof *stats);
            CUDA_TRY(cudaEventElapsedTime(&stats->ms_total, ctx->ev[0], ctx->ev[1]));
            stats->paths = paths;
            stats->rays = rays;
            stats->launches = launches;
            stats->iterations = iterations;
        }
        return RT_OK;
    }();
    cudaFreeAsync(base, stream);
    return st;
}

} // namespace

extern "C" {

rt_status rt_adaptive_error_device(rt_context* ctx, const void* planes_dev, int32_t width, int32_t height, void* error_dev) try {
    ARG_CHECK(ctx && planes_dev && error_dev, "ctx/planes_dev/error_dev is NULL");
    ARG_CHECK(width > 0 && height > 0, "width/height must be positive");
    ARG_CHECK(uint64_t(width) * uint64_t(height) < (1ull << 31), "frame has more than 2^31 pixels");
    rt_status st = make_current(ctx);
    if (st != RT_OK) return st;
    float* e = nullptr;
    CUDA_TRY(rtd::malloc_async(&e, size_t(width) * size_t(height) * sizeof(float), ctx->stream));
    rtd::launch_adapt_error_map(static_cast<const float4*>(planes_dev), width, height, e, static_cast<float*>(error_dev), ctx->stream);
    const cudaError_t err = cudaGetLastError();
    cudaFreeAsync(e, ctx->stream);
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
    if ((st = ensure_accum(ctx, npix)) != RT_OK) return st;
    if ((st = ensure_out(ctx, npix)) != RT_OK) return st;
    rt_stats local;
    if ((st = adaptive_into(ctx, scene, p, a, ctx->accum, nullptr, nullptr, &local)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    rtd::launch_tonemap(ctx->accum, p->width, p->height, ctx->out_rgb, nullptr, ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_rgb, ctx->out_rgb, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    std::vector<float4> acc(out_spp ? npix : 0);
    if (out_spp) CUDA_TRY(cudaMemcpyAsync(acc.data(), ctx->accum, npix * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < acc.size(); ++i) out_spp[i] = int32_t(acc[i].w); // (exact: counts stay below 2^24)
    CUDA_TRY(cudaEventElapsedTime(&local.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_d2h, ctx->ev[2], ctx->ev[3]));
    local.launches += 1;
    if (stats) *stats = local;
    return RT_OK;
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
    rtd::DCamera* d_cams = nullptr;
    CUDA_TRY(rtd::malloc_async(&d_cams, cams.size() * sizeof(rtd::DCamera), ctx->stream));
    const rt_status st = [&]() -> rt_status {
        CUDA_TRY(cudaMemcpyAsync(d_cams, cams.data(), cams.size() * sizeof(rtd::DCamera), cudaMemcpyHostToDevice, ctx->stream));
        rtd::DRenderParams rp = to_device_params(*p);
        rp.spp = p->spp * n_frames; // <= 2^31 - 1: check_frames
        rp.frame_cams = d_cams;
        rp.div_spp = rtd::make_fastdiv(uint32_t(p->spp));
        return render_rp(ctx, scene, rp, p->pipeline, accum, stats);
    }();
    cudaFreeAsync(d_cams, ctx->stream);
    return st;
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
    if ((st = ensure_accum(ctx, total)) != RT_OK) return st;
    if ((st = ensure_out(ctx, total)) != RT_OK) return st;
    CUDA_TRY(cudaMemsetAsync(ctx->accum, 0, total * sizeof(float4), ctx->stream));
    rt_stats local;
    if ((st = frames_into(ctx, scene, p, cameras, n_frames, ctx->accum, &local)) != RT_OK) return st;
    CUDA_TRY(cudaEventRecord(ctx->ev[1], ctx->stream));
    for (int32_t f = 0; f < n_frames; ++f)
        rtd::launch_tonemap(ctx->accum + size_t(f) * npix, p->width, p->height, ctx->out_rgb + size_t(f) * npix * 3, nullptr,
                            ctx->sm_count, ctx->stream);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev[2], ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_rgb, ctx->out_rgb, total * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaEventRecord(ctx->ev[3], ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_tonemap, ctx->ev[1], ctx->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&local.ms_d2h, ctx->ev[2], ctx->ev[3]));
    local.launches += uint32_t(n_frames);
    if (stats) *stats = local;
    return RT_OK;
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
    float* d_out = nullptr;
    CUDA_TRY(rtd::malloc_async(&d_out, n * sizeof(float), ctx->stream));
    cudaError_t e = rtd::jpeg_pixels_device(img, d_out, ctx->stream, ms_device);
    float* host = e == cudaSuccess ? static_cast<float*>(malloc(n * sizeof(float))) : nullptr;
    if (e == cudaSuccess && host) {
        e = cudaMemcpyAsync(host, d_out, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    }
    cudaFreeAsync(d_out, ctx->stream);
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
