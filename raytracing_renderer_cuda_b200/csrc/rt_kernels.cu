// rt_kernels.cu — parity hook, per-path megakernel, tonemap.  sm_100a only.
#include <cstdlib>

#include "rt_kernels.cuh"
#include "rt_shade.cuh"

namespace rtd {

// --------------------------------------------------------------- trace_primary ----
// scene.hit(r, tmin, FLT_MAX, rec) for caller-supplied rays (hitable_list.h:60-79).
__global__ void __launch_bounds__(256) k_trace_primary(const __grid_constant__ DScene sc, const rt_ray* __restrict__ rays,
                                                       size_t n, float tmin, int use_bvh, rt_hit* __restrict__ hits) {
    size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rt_ray in = rays[i];
    Ray r;
    r.o = mk(in.origin[0], in.origin[1], in.origin[2]);
    r.d = mk(in.direction[0], in.direction[1], in.direction[2]);
    r.time = in.time;
    RayQ q = make_rayq(r);
    Hit h = (use_bvh == 3 && sc.nodes4q) ? closest_hit_bvh4<true>(sc, q, tmin)
            : (use_bvh == 2 && sc.nodes4)  ? closest_hit_bvh4<false>(sc, q, tmin)
                                           : closest_hit(sc, q, tmin, use_bvh != 0);
    rt_hit out;
    if (h.prim == RT_INVALID_ID) {
        out.t = FLT_MAX;
        out.id = RT_INVALID_ID;
        out.p[0] = out.p[1] = out.p[2] = 0.f;
        out.n[0] = out.n[1] = out.n[2] = 0.f;
        out.u = out.v = 0.f;
    } else {
        V3 p, nn;
        hit_surface(sc, q, h, p, nn);
        out.t = h.t;
        out.id = __ldg(&sc.sph_c[h.prim]).z;
        out.p[0] = p.x; out.p[1] = p.y; out.p[2] = p.z;
        out.n[0] = nn.x; out.n[1] = nn.y; out.n[2] = nn.z;
        sphere_uv(nn, out.u, out.v);
    }
    hits[i] = out;
}

void launch_trace_primary(const DScene& sc, const rt_ray* rays_dev, size_t n, float tmin, int use_bvh,
                          rt_hit* hits_dev, cudaStream_t st) {
    if (n == 0) return;
    unsigned blocks = unsigned((n + 255) / 256);
    k_trace_primary<<<blocks, 256, 0, st>>>(sc, rays_dev, n, tmin, use_bvh, hits_dev);
}

// --------------------------------------------------------------- shade_probe ----
__global__ void __launch_bounds__(256) k_shade_probe(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp,
                                                     const rt_ray* __restrict__ rays, size_t n, int use_bvh,
                                                     rt_shade_sample* __restrict__ out) {
    extern __shared__ __align__(16) uint32_t smem[];
    perlin_stage(smem, threadIdx.x, blockDim.x);
    __syncthreads();
    PerlinTab pt{smem, threadIdx.x & 31u};
    size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rt_ray in = rays[i];
    Ray r;
    r.o = mk(in.origin[0], in.origin[1], in.origin[2]);
    r.d = mk(in.direction[0], in.direction[1], in.direction[2]);
    r.time = in.time;
    RayQ q = make_rayq(r);
    Hit h = closest_hit(sc, q, rp.tmin, use_bvh != 0);
    rt_shade_sample o;
    memset(&o, 0, sizeof o);
    o.id = RT_INVALID_ID;
    if (h.prim != RT_INVALID_ID) {
        V3 E, att;
        Ray next;
        next.o = next.d = mk(0.f, 0.f, 0.f);
        next.time = 0.f;
        V3 direct = mk(0.f, 0.f, 0.f); // the probe evaluates the reference estimator: the host entry clears rp.flags
        bool nee_vertex;
        uint32_t shadow_rays = 0;
        bool cont = shade_terms(sc, rp, pt, q, h, uint32_t(i), 0u, 1u, E, att, next, direct, nee_vertex, shadow_rays);
        o.id = __ldg(&sc.sph_c[h.prim]).z;
        o.continues = cont ? 1u : 0u;
        o.t = h.t;
        o.emitted[0] = E.x; o.emitted[1] = E.y; o.emitted[2] = E.z;
        o.attenuation[0] = att.x; o.attenuation[1] = att.y; o.attenuation[2] = att.z;
        if (cont) {
            o.scattered.origin[0] = next.o.x; o.scattered.origin[1] = next.o.y; o.scattered.origin[2] = next.o.z;
            o.scattered.direction[0] = next.d.x; o.scattered.direction[1] = next.d.y; o.scattered.direction[2] = next.d.z;
            o.scattered.time = next.time;
        }
    }
    out[i] = o;
}

void launch_shade_probe(const DScene& sc, const DRenderParams& rp, const rt_ray* rays_dev, size_t n, bool use_bvh,
                        rt_shade_sample* out_dev, cudaStream_t st) {
    if (n == 0) return;
    const size_t smem = RT_PERLIN_SMEM_WORDS * sizeof(uint32_t);
    static_assert(RT_PERLIN_SMEM_WORDS * sizeof(uint32_t) <= 48u * 1024u, "needs cudaFuncAttributeMaxDynamicSharedMemorySize (per device)");
    k_shade_probe<<<unsigned((n + 255) / 256), 256, smem, st>>>(sc, rp, rays_dev, n, use_bvh ? 1 : 0, out_dev);
}

// --------------------------------------------------------------- megakernel ----
// One thread per path, grid-stride over (sample, pixel) with pixel fastest so a warp
// covers 32 neighbouring pixels of one sample.  This is the reference's structure
// (render + color(), main.cu:35-74,97-132) on the flat scene; it is kept as the
// RT_PIPE_MEGAKERNEL pipeline and as the yardstick the wavefront pipeline is measured against.
// RM_ADAPT: adaptive sampling, path -> pixel rp.adapt_pixels[path mod n] (n = div_npix.d), values into the sample's parity plane.
// RM_FRAMES: a frame sequence, the camera and the accumulator of the sample's frame (DRenderParams::frame_cams).
template <int RM>
__global__ void __launch_bounds__(256) k_render_mega(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp,
                                                     int use_bvh, float4* __restrict__ accum,
                                                     unsigned long long* __restrict__ ray_counter) {
    extern __shared__ __align__(16) uint32_t smem[];
    perlin_stage(smem, threadIdx.x, blockDim.x);
    __syncthreads();
    PerlinTab pt{smem, threadIdx.x & 31u};

    const unsigned long long npix = RM == RM_ADAPT ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    const unsigned long long npaths = npix * (unsigned long long)rp.spp;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long nrays = 0;
    for (unsigned long long path = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; path < npaths; path += stride) {
        uint32_t pixel = uint32_t(path % npix);
        if (RM == RM_ADAPT) pixel = __ldg(rp.adapt_pixels + pixel);
        uint32_t sample = uint32_t(path / npix) + uint32_t(rp.sample_offset);
        Ray r = camera_ray<RM>(sc, rp, pixel, sample);
        V3 A = mk(rp.world_r, rp.world_g, rp.world_b); // main.cu:40
        V3 result = mk(0.f, 0.f, 0.f);                 // exceeded recursion (main.cu:70)
        V3 direct = mk(0.f, 0.f, 0.f);                 // shadow/emission rays of the path (RT_RENDER_EMITTER_SAMPLING)
        bool nee_vertex = false;                       // the ray being traced left a lambertian hit that traced one
        uint32_t shadow_rays = 0;
        for (int bounce = 1; bounce <= rp.max_depth; ++bounce) {
            RayQ q = make_rayq(r);
            Hit h = closest_hit(sc, q, rp.tmin, use_bvh != 0);
            ++nrays;
            if (h.prim == RT_INVALID_ID) { // main.cu:66-67: return world colour times nothing: A itself
                result = A;
                break;
            }
            Ray next;
            if (nee_vertex && is_listed_emitter(sc, h.prim)) { // counted by the shadow ray of the previous hit
                result = mk(0.f, 0.f, 0.f);
                break;
            }
            if (!shade_hit(sc, rp, pt, q, h, pixel, sample, uint32_t(bounce), A, next, direct, nee_vertex, shadow_rays)) {
                result = A;
                break;
            }
            r = next;
        }
        nrays += shadow_rays;
        atomicAdd(&accum_plane<RM>(accum, rp, sample)[pixel], make_float4(result.x + direct.x, result.y + direct.y, result.z + direct.z, 1.f)); // RED.E.ADD.F32x4 (sm_90+)
    }
    // one counter update per warp
    for (int off = 16; off > 0; off >>= 1) nrays += __shfl_down_sync(0xffffffffu, nrays, off);
    if ((threadIdx.x & 31) == 0 && nrays) atomicAdd(ray_counter, nrays);
}

void launch_render_mega(const DScene& sc, const DRenderParams& rp, bool use_bvh, float4* accum,
                        unsigned long long* ray_counter, int sm_count, cudaStream_t st) {
    const unsigned long long npix = rp.adapt_pixels ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    unsigned long long npaths = npix * (unsigned long long)rp.spp;
    if (npaths == 0) return;
    const size_t smem = RT_PERLIN_SMEM_WORDS * sizeof(uint32_t);
    unsigned long long want = (npaths + 255) / 256;
    unsigned long long cap = (unsigned long long)sm_count * 32; // several waves of resident CTAs, grid-stride beyond
    unsigned blocks = unsigned(want < cap ? want : cap);
    if (rp.adapt_pixels) k_render_mega<RM_ADAPT><<<blocks, 256, smem, st>>>(sc, rp, use_bvh ? 1 : 0, accum, ray_counter);
    else if (rp.frame_cams) k_render_mega<RM_FRAMES><<<blocks, 256, smem, st>>>(sc, rp, use_bvh ? 1 : 0, accum, ray_counter);
    else k_render_mega<RM_PLAIN><<<blocks, 256, smem, st>>>(sc, rp, use_bvh ? 1 : 0, accum, ray_counter);
}

// --------------------------------------------------------------- tonemap ----
// main.cu:124-127: col /= spp (vec3::operator/=(float): rz(1/f) then RZ multiplies,
// vec3.h:138-151), saturate (vec3.h:349-356), gamma 2 = __fsqrt_rz (vec3.h:181-187).
// out_rgb: reference framebuffer layout, index j*W+i with j = 0 the bottom row.
// out_rgb8: the writer loop main.cu:476-487 — Y flip and int(255.999f*c) & 255.
// Pixel finalisation of main.cu:124-127 (+ the writer's conversion, main.cu:476-487) for G consecutive pixels of one row.
// G = 4 when the width allows it: four 16-byte loads, three 16-byte stores of float RGB, three 4-byte stores of rgb8 per
// thread — the pass is pure streaming (16 B read + 15 B written per pixel) and the per-pixel index division and byte
// stores of the scalar form kept it at 74 % of the copy bandwidth at 8K (profiles/r02_framebuffer_passes.md).
struct Rgb {
    float r, g, b;
};
RT_DEV Rgb finalise(float4 a) {
    const float inv = div_rz(1.0f, a.w);
    return Rgb{sqrt_rz(__saturatef(__fmul_rz(a.x, inv))), sqrt_rz(__saturatef(__fmul_rz(a.y, inv))), sqrt_rz(__saturatef(__fmul_rz(a.z, inv)))};
}
RT_DEV uint32_t q8(float c) { return uint32_t(int(255.999f * c) & 255); }
template <int G>
RT_DEV void store_pixels(const Rgb (&px)[G], size_t idx, int width, int height, const FastDiv& div_w, float* __restrict__ out_rgb,
                         uint8_t* __restrict__ out_rgb8) {
    if (out_rgb) {
        if (G == 4) {
            float4* o = reinterpret_cast<float4*>(out_rgb + idx * 3);
            o[0] = make_float4(px[0].r, px[0].g, px[0].b, px[1].r);
            o[1] = make_float4(px[1].g, px[1].b, px[2].r, px[2].g);
            o[2] = make_float4(px[2].b, px[3].r, px[3].g, px[3].b);
        } else {
#pragma unroll
            for (int k = 0; k < G; ++k) {
                out_rgb[(idx + k) * 3 + 0] = px[k].r;
                out_rgb[(idx + k) * 3 + 1] = px[k].g;
                out_rgb[(idx + k) * 3 + 2] = px[k].b;
            }
        }
    }
    if (out_rgb8) { // Y flip: row j of the frame is row height - 1 - j of the picture
        const uint32_t j = fastdiv(uint32_t(idx), div_w), i = uint32_t(idx) - j * uint32_t(width);
        const size_t rev = (size_t(height) - 1 - j) * size_t(width) + i;
        if (G == 4) {
            uint32_t* o = reinterpret_cast<uint32_t*>(out_rgb8 + rev * 3);
            o[0] = q8(px[0].r) | q8(px[0].g) << 8 | q8(px[0].b) << 16 | q8(px[1].r) << 24;
            o[1] = q8(px[1].g) | q8(px[1].b) << 8 | q8(px[2].r) << 16 | q8(px[2].g) << 24;
            o[2] = q8(px[2].b) | q8(px[3].r) << 8 | q8(px[3].g) << 16 | q8(px[3].b) << 24;
        } else {
#pragma unroll
            for (int k = 0; k < G; ++k) {
                out_rgb8[(rev + k) * 3 + 0] = uint8_t(q8(px[k].r));
                out_rgb8[(rev + k) * 3 + 1] = uint8_t(q8(px[k].g));
                out_rgb8[(rev + k) * 3 + 2] = uint8_t(q8(px[k].b));
            }
        }
    }
}
template <int G>
__global__ void __launch_bounds__(256) k_tonemap(const float4* __restrict__ accum, int width, int height, const __grid_constant__ FastDiv div_w,
                                                 float* __restrict__ out_rgb, uint8_t* __restrict__ out_rgb8) {
    const size_t ngroups = size_t(width) * height / G;
    for (size_t g = size_t(blockIdx.x) * blockDim.x + threadIdx.x; g < ngroups; g += size_t(gridDim.x) * blockDim.x) {
        const size_t idx = g * G;
        Rgb px[G];
#pragma unroll
        for (int k = 0; k < G; ++k) px[k] = finalise(__ldg(&accum[idx + k]));
        store_pixels<G>(px, idx, width, height, div_w, out_rgb, out_rgb8);
    }
}

// Grid of a grid-stride streaming pass over `items` work items, 256 threads per CTA: exactly the CTAs that are resident at
// once (SMs x occupancy of THIS kernel), so the pass has one wave and no partial second one (k_reduce_tonemap<4> holds
// 5 CTAs per SM at 44 registers; a grid of 8 per SM ran 1.6 waves), or fewer when the frame is small.
template <typename K>
static unsigned stream_grid(K kernel, size_t items, int sm_count) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, 256, 0) != cudaSuccess || per_sm < 1) per_sm = 4;
    const size_t want = (items + 255) / 256, cap = size_t(sm_count > 0 ? sm_count : 1) * size_t(per_sm);
    const size_t n = want < cap ? want : cap;
    return unsigned(n ? n : 1);
}

// --------------------------------------------------------------- fused reduce + tonemap ----
// Multi-GPU pixel finalisation in ONE kernel over NVLink peer memory: sums the float4 accumulators of all
// ranks for a band of rows and applies main.cu:124-127 (+ the writer conversion) to the sum.  Two ways to
// form the sum:
//   * multicast != nullptr: one `multimem.ld_reduce.global.add.v4.f32` per pixel on the NVLS multicast
//     address of the symmetric accumulator — the NVSwitch adds the G copies in the fabric and returns the sum;
//   * otherwise: G `ld.global` loads from the peers' mapped accumulators, added in rank order (bit-reproducible).
// The outputs may themselves be peer pointers (each rank writes its band straight into the root's image).
struct PeerPtrs {
    const float4* p[16];
};
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float4* mc) {
    float4 v;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(mc)
                 : "memory");
    return v;
}
template <int G>
__global__ void __launch_bounds__(256) k_reduce_tonemap(const __grid_constant__ PeerPtrs peers, int n_peers,
                                                        const float4* __restrict__ multicast, int width, int height,
                                                        const __grid_constant__ FastDiv div_w, int row_begin, int row_end,
                                                        float* __restrict__ out_rgb, uint8_t* __restrict__ out_rgb8, float4* __restrict__ out_sum) {
    const size_t first = size_t(row_begin) * size_t(width) / G, last = size_t(row_end) * size_t(width) / G;
    for (size_t g = first + size_t(blockIdx.x) * blockDim.x + threadIdx.x; g < last; g += size_t(gridDim.x) * blockDim.x) {
        const size_t idx = g * G;
        Rgb px[G];
#pragma unroll
        for (int k = 0; k < G; ++k) {
            float4 a;
            if (multicast) {
                a = multimem_ld_reduce_add(multicast + idx + k);
            } else {
                a = __ldcg(&peers.p[0][idx + k]); // (L2 only: a peer's accumulator changes from frame to frame)
                for (int m = 1; m < n_peers; ++m) {
                    const float4 b = __ldcg(&peers.p[m][idx + k]);
                    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
                }
            }
            if (out_sum) out_sum[idx + k] = a;
            px[k] = finalise(a);
        }
        store_pixels<G>(px, idx, width, height, div_w, out_rgb, out_rgb8);
    }
}

void launch_reduce_tonemap(const void* const* peer_accum, int n_peers, const void* multicast, int width, int height,
                           int row_begin, int row_end, float* out_rgb, uint8_t* out_rgb8, float4* out_sum, int sm_count,
                           cudaStream_t st) {
    if (row_end <= row_begin || width <= 0) return;
    PeerPtrs pp{};
    if (peer_accum) // (NULL with a multicast address: the kernel then never reads the table)
        for (int k = 0; k < n_peers && k < 16; ++k) pp.p[k] = static_cast<const float4*>(peer_accum[k]);
    const size_t npix = size_t(row_end - row_begin) * size_t(width);
    const FastDiv div_w = make_fastdiv(uint32_t(width));
    // Four pixels per thread give 16-byte stores, but a warp's loads of one pixel slot then touch every other 16 bytes of 2 KB:
    // fine from local HBM, half-used 32-byte requests over NVLink.  With peers (or RT_REDUCE_G=1) one pixel per thread: a warp
    // reads 512 contiguous bytes of every member (A/B: profiles/r02_framebuffer_passes.md).
    const char* g_env = getenv("RT_REDUCE_G");
    const bool wide = g_env ? g_env[0] == '4' : (n_peers <= 1 && multicast == nullptr);
    if (wide && width % 4 == 0 && uintptr_t(out_rgb) % 16 == 0 && uintptr_t(out_rgb8) % 4 == 0) // (vector stores need the alignment)
        k_reduce_tonemap<4><<<stream_grid(k_reduce_tonemap<4>, npix / 4, sm_count), 256, 0, st>>>(
            pp, n_peers, static_cast<const float4*>(multicast), width, height, div_w, row_begin, row_end, out_rgb, out_rgb8, out_sum);
    else
        k_reduce_tonemap<1><<<stream_grid(k_reduce_tonemap<1>, npix, sm_count), 256, 0, st>>>(
            pp, n_peers, static_cast<const float4*>(multicast), width, height, div_w, row_begin, row_end, out_rgb, out_rgb8, out_sum);
}

// --------------------------------------------------------------- self-test of the arithmetic helpers ----
__global__ void k_selftest_rz(const float* __restrict__ x, const float* __restrict__ y, size_t n, float* __restrict__ out) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x) {
        out[4 * i + 0] = div_rz(x[i], y[i]);
        out[4 * i + 1] = __fdiv_rz(x[i], y[i]);
        out[4 * i + 2] = sqrt_rz(x[i]);
        out[4 * i + 3] = __fsqrt_rz(x[i]);
    }
}
void launch_selftest_rz(const float* x, const float* y, size_t n, float* out, cudaStream_t st) {
    if (n) k_selftest_rz<<<1024, 256, 0, st>>>(x, y, n, out);
}

void launch_tonemap(const float4* accum, int width, int height, float* out_rgb, uint8_t* out_rgb8, int sm_count, cudaStream_t st) {
    const size_t npix = size_t(width) * height;
    if (npix == 0) return;
    const FastDiv div_w = make_fastdiv(uint32_t(width));
    if (width % 4 == 0 && uintptr_t(out_rgb) % 16 == 0 && uintptr_t(out_rgb8) % 4 == 0)
        k_tonemap<4><<<stream_grid(k_tonemap<4>, npix / 4, sm_count), 256, 0, st>>>(accum, width, height, div_w, out_rgb, out_rgb8);
    else
        k_tonemap<1><<<stream_grid(k_tonemap<1>, npix, sm_count), 256, 0, st>>>(accum, width, height, div_w, out_rgb, out_rgb8);
}

__global__ void __launch_bounds__(256) k_rgb_to_rgba(const float* __restrict__ rgb, float4* __restrict__ rgba, size_t n) {
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += size_t(gridDim.x) * blockDim.x)
        rgba[i] = make_float4(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2], 1.f);
}

void launch_rgb_to_rgba(const float* rgb, float4* rgba, size_t n_texels, int sm_count, cudaStream_t st) {
    if (n_texels == 0) return;
    size_t want = (n_texels + 255) / 256;
    const size_t cap = size_t(sm_count > 0 ? sm_count : 1) * 16u;
    unsigned blocks = unsigned(want < cap ? want : cap);
    k_rgb_to_rgba<<<blocks, 256, 0, st>>>(rgb, rgba, n_texels);
}

} // namespace rtd
