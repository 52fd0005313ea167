// rt_kernels.cuh — host-callable launchers of the sm_100a kernels (defined in the .cu files).
#pragma once

#include <cuda_runtime.h>

#include "rt_device.cuh"

namespace rtd {

// Stream-ordered scratch and scene memory comes from the calling context's OWN memory pool (rt_api.cu creates one per
// context with an unlimited release threshold; make_current() selects it for the calling thread): freed blocks are
// reused by the next scene instead of going back to the driver, and the device's default pool — shared with torch and
// every other user of cudaMallocAsync in the process — is left alone.
void set_thread_mempool(cudaMemPool_t pool);
cudaError_t malloc_async_bytes(void** p, size_t bytes, cudaStream_t st);
template <class T>
inline cudaError_t malloc_async(T** p, size_t bytes, cudaStream_t st) {
    return malloc_async_bytes(reinterpret_cast<void**>(p), bytes, st);
}

// Scratch of `count` T from malloc_async, freed on the same stream when the buffer goes out of scope (stream order makes
// the free wait for the work queued before it, so no exit path needs a synchronisation or a hand-written free).
template <class T>
class PoolBuffer {
  public:
    PoolBuffer() = default;
    PoolBuffer(PoolBuffer&& o) noexcept : p_(o.p_), st_(o.st_) { o.p_ = nullptr; }
    ~PoolBuffer() {
        if (p_) cudaFreeAsync(p_, st_);
    }
    cudaError_t alloc(size_t count, cudaStream_t st) { // on an empty buffer
        st_ = st;
        const cudaError_t e = malloc_async(&p_, count * sizeof(T), st);
        if (e != cudaSuccess) p_ = nullptr;
        return e;
    }
    T* get() const { return p_; }
    T* release() { // the caller frees the memory from now on
        T* p = p_;
        p_ = nullptr;
        return p;
    }

  private:
    T* p_ = nullptr;
    cudaStream_t st_ = nullptr;
};

// A timing event destroyed when it goes out of scope
struct TimingEvent {
    cudaEvent_t ev = nullptr;
    TimingEvent() = default;
    TimingEvent(const TimingEvent&) = delete;
    TimingEvent& operator=(const TimingEvent&) = delete;
    ~TimingEvent() {
        if (ev) cudaEventDestroy(ev);
    }
    cudaError_t create() { return cudaEventCreate(&ev); }
};

// returns a failing cudaError_t from a function that returns one (its PoolBuffers and TimingEvents release themselves)
#define RTD_TRY(expr)                          \
    do {                                       \
        const cudaError_t e__ = (expr);        \
        if (e__ != cudaSuccess) return e__;    \
    } while (0)

// parity hook: closest hit for caller-supplied rays
void launch_trace_primary(const DScene& sc, const rt_ray* rays_dev, size_t n, float tmin, int use_bvh, // 0 list, 1 BVH, 2 4-wide BVH
                          rt_hit* hits_dev, cudaStream_t st);

// parity hook: closest hit + one shading step (terms of main.cu:45-55) per caller-supplied ray
void launch_shade_probe(const DScene& sc, const DRenderParams& rp, const rt_ray* rays_dev, size_t n, bool use_bvh,
                        rt_shade_sample* out_dev, cudaStream_t st);

// one thread runs whole paths (reference structure, main.cu:35-74,97-132)
void launch_render_mega(const DScene& sc, const DRenderParams& rp, bool use_bvh, float4* accum,
                        unsigned long long* ray_counter, int sm_count, cudaStream_t st);

// pixel finalisation (main.cu:124-127) + optional writer conversion (main.cu:476-487)
void launch_tonemap(const float4* accum, int width, int height, float* out_rgb, uint8_t* out_rgb8, int sm_count, cudaStream_t st);

// multi-GPU: sum of the peers' accumulators (peer loads or NVLS multimem.ld_reduce) fused with the tonemap
void launch_reduce_tonemap(const void* const* peer_accum, int n_peers, const void* multicast, int width, int height,
                           int row_begin, int row_end, float* out_rgb, uint8_t* out_rgb8, float4* out_sum, int sm_count, cudaStream_t st);

// denoiser (rt_denoise.cu): first-hit features of feature_spp camera samples per pixel (2 float4 planes of width*height),
// and one level of the edge-avoiding à-trous filter (taps 2^level apart); from_accum: `in` is a render's accumulator
void launch_features(const DScene& sc, const DRenderParams& rp, bool use_bvh, int feature_spp, float4* features, cudaStream_t st);
void launch_atrous(const float4* in, bool from_accum, const float4* features, int width, int height, int level, float sigma_color,
                   float sigma_normal, float sigma_depth, float sigma_albedo, float4* out, cudaStream_t st);

// adaptive sampling (rt_adaptive.cu).  planes: two float4 planes of width*height (A: even samples, B: odd samples).
// Windowed error map of the planes into ebar (e_scratch: width*height floats)
void launch_adapt_error_map(const float4* planes, int width, int height, float* e_scratch, float* ebar, cudaStream_t st);
// uint32 words of scratch launch_adapt_select needs besides e_scratch
size_t adapt_select_scratch_words(uint32_t npix);
// next = the entries of list (n pixels) whose windowed error is >= tau and whose count is < max_spp, in list order; *n_next
// (device) = their number; *launches = kernels launched
cudaError_t launch_adapt_select(const float4* planes, int width, int height, const uint32_t* list, uint32_t n, float tau,
                                int32_t max_spp, float* e_scratch, uint32_t* words, uint32_t* next, uint32_t* n_next, uint32_t* launches,
                                cudaStream_t st);
void launch_adapt_iota(uint32_t* list, uint32_t n, cudaStream_t st);
// accum = A + B (written, not added)
void launch_adapt_merge(const float4* planes, uint32_t npix, float4* accum, cudaStream_t st);

// self-test: out[4i..4i+3] = div_rz(x, y), __fdiv_rz(x, y), sqrt_rz(x), __fsqrt_rz(x)  (rt_device.cuh)
void launch_selftest_rz(const float* x_dev, const float* y_dev, size_t n, float* out_dev, cudaStream_t st);

// float RGB (w*h*3) -> float4 RGBA staging for the image-texture cudaArray
void launch_rgb_to_rgba(const float* rgb, float4* rgba, size_t n_texels, int sm_count, cudaStream_t st);

// wavefront pipeline state (rt_wavefront.cu)
struct WavefrontState;
WavefrontState* wavefront_create(size_t pool_paths, cudaStream_t st);
void wavefront_destroy(WavefrontState* ws);
size_t wavefront_pool(const WavefrontState* ws);
// renders rp.spp samples of every pixel into accum (+=); returns launches/iterations.  false: the frame did not
// finish within the iteration bound (a defect or a CUDA error — never a silently short frame)
bool wavefront_render(WavefrontState* ws, const DScene& sc, const DRenderParams& rp, bool use_bvh, float4* accum,
                      unsigned long long* ray_counter, int sm_count, cudaStream_t st, uint32_t* launches,
                      uint32_t* iterations);

} // namespace rtd
