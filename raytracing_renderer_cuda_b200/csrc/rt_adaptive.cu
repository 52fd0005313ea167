// rt_adaptive.cu — adaptive sampling: the per-pixel noise estimate of a two-plane accumulator and the device step that
// decides which pixels keep sampling.  The passes themselves are the ADAPT instantiations of the render kernels
// (rt_wavefront.cu, rt_kernels.cu): a path adds into plane A (even samples, counted from the first sample of the adaptive
// render) or plane B (odd samples), W*H float4 apart.  sm_100a only.
//
// Error of pixel p, with g(x) = sqrt(saturate(x)) the display transform of the finalisation:
//   e_p = (|g(A_r/A_w) - g(B_r/B_w)| + |g(A_g/A_w) - g(B_g/B_w)| + |g(A_b/A_w) - g(B_b/B_w)|) / 6     (+inf if A_w or B_w is 0)
// i.e. half the mean over the channels of the difference of the two half means: an estimate of the standard error of the
// full mean in display space.  Windowed error: ebar_p = (sum of e over the 3x3 neighbourhood, coordinates clamped to the
// frame, added in row-major order) / 9.  Every operation is one IEEE round-to-nearest float operation (the Makefile's
// flags give -prec-div / -prec-sqrt and no expression here can contract into an FMA), so a numpy float32 restatement
// reproduces the values bit for bit (tests/test_adaptive.py).
#include "rt_kernels.cuh"
#include "rt_prims.cuh"

namespace rtd {

RT_DEV float display(float sum, float w) { return sqrtf(__saturatef(sum / w)); }

__global__ void __launch_bounds__(256) k_adapt_error(const float4* __restrict__ planes, uint32_t npix, float* __restrict__ e) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const float4 a = __ldg(&planes[p]), b = __ldg(&planes[size_t(npix) + p]);
    float v = __int_as_float(0x7f800000); // +inf: a plane without samples
    if (a.w > 0.f && b.w > 0.f) {
        const float dr = fabsf(display(a.x, a.w) - display(b.x, b.w));
        const float dg = fabsf(display(a.y, a.w) - display(b.y, b.w));
        const float db = fabsf(display(a.z, a.w) - display(b.z, b.w));
        v = (dr + dg + db) / 6.f;
    }
    e[p] = v;
}

// Entry i of the list (pixel list[i]; list == nullptr: pixel i): the windowed error, and whether the pixel keeps sampling,
// ebar >= tau and fewer than max_spp samples so far.  keep / ebar may be nullptr.
__global__ void __launch_bounds__(256) k_adapt_select(const float* __restrict__ e, const float4* __restrict__ planes, int width,
                                                      int height, const uint32_t* __restrict__ list, uint32_t n, float tau,
                                                      float max_spp, uint32_t* __restrict__ keep, float* __restrict__ ebar) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = list ? __ldg(&list[i]) : i;
    const int y = int(p / uint32_t(width)), x = int(p - uint32_t(y) * uint32_t(width));
    float s = 0.f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int yy = min(max(y + dy, 0), height - 1);
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int xx = min(max(x + dx, 0), width - 1);
            s = s + __ldg(&e[size_t(yy) * size_t(width) + size_t(xx)]);
        }
    }
    const float m = s / 9.f;
    if (ebar) ebar[p] = m;
    if (keep) {
        const size_t npix = size_t(width) * size_t(height);
        const float count = __ldg(&planes[p]).w + __ldg(&planes[npix + p]).w;
        keep[i] = (m >= tau && count < max_spp) ? 1u : 0u;
    }
}

// next[pos[i]] = list[i] for the kept entries (pos = exclusive sum of keep: list order is kept); *n_next = entries kept
__global__ void __launch_bounds__(256) k_adapt_compact(const uint32_t* __restrict__ list, const uint32_t* __restrict__ keep,
                                                       const uint32_t* __restrict__ pos, uint32_t n, uint32_t* __restrict__ next,
                                                       uint32_t* __restrict__ n_next) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = __ldg(&keep[i]), at = __ldg(&pos[i]);
    if (k) next[at] = __ldg(&list[i]);
    if (i == n - 1u) *n_next = at + k;
}

__global__ void __launch_bounds__(256) k_adapt_iota(uint32_t* __restrict__ list, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) list[i] = i;
}

__global__ void __launch_bounds__(256) k_adapt_merge(const float4* __restrict__ planes, uint32_t npix, float4* __restrict__ accum) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const float4 a = __ldg(&planes[p]), b = __ldg(&planes[size_t(npix) + p]);
    accum[p] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

static unsigned blocks_of(uint32_t n) { return (n + 255u) / 256u; }

void launch_adapt_error_map(const float4* planes, int width, int height, float* e_scratch, float* ebar, cudaStream_t st) {
    const uint32_t npix = uint32_t(width) * uint32_t(height);
    k_adapt_error<<<blocks_of(npix), 256, 0, st>>>(planes, npix, e_scratch);
    k_adapt_select<<<blocks_of(npix), 256, 0, st>>>(e_scratch, planes, width, height, nullptr, npix, 0.f, 0.f, nullptr, ebar);
}

size_t adapt_select_scratch_words(uint32_t npix) { return 2 * size_t(npix) + prims::scan_scratch_elems(npix); }

// kernel launches of prims::exclusive_sum over n values
static uint32_t scan_launches(size_t n) {
    if (n == 0) return 0;
    const size_t tiles = (n + prims::kTile - 1) / prims::kTile;
    return tiles == 1 ? 1u : 2u + scan_launches(tiles);
}

cudaError_t launch_adapt_select(const float4* planes, int width, int height, const uint32_t* list, uint32_t n, float tau,
                                int32_t max_spp, float* e_scratch, uint32_t* words, uint32_t* next, uint32_t* n_next, uint32_t* launches,
                                cudaStream_t st) {
    *launches = 3u + scan_launches(n);
    const uint32_t npix = uint32_t(width) * uint32_t(height);
    uint32_t* keep = words;
    uint32_t* pos = words + npix;
    uint32_t* scan = words + 2 * size_t(npix);
    k_adapt_error<<<blocks_of(npix), 256, 0, st>>>(planes, npix, e_scratch);
    k_adapt_select<<<blocks_of(n), 256, 0, st>>>(e_scratch, planes, width, height, list, n, tau, float(max_spp), keep, nullptr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if ((e = prims::exclusive_sum<uint32_t>(keep, pos, n, scan, st)) != cudaSuccess) return e;
    k_adapt_compact<<<blocks_of(n), 256, 0, st>>>(list, keep, pos, n, next, n_next);
    return cudaGetLastError();
}

void launch_adapt_iota(uint32_t* list, uint32_t n, cudaStream_t st) { k_adapt_iota<<<blocks_of(n), 256, 0, st>>>(list, n); }

void launch_adapt_merge(const float4* planes, uint32_t npix, float4* accum, cudaStream_t st) {
    k_adapt_merge<<<blocks_of(npix), 256, 0, st>>>(planes, npix, accum);
}

} // namespace rtd
