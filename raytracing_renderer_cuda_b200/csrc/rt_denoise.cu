// rt_denoise.cu — denoiser: first-hit feature buffers and the edge-avoiding à-trous wavelet filter (Dammertz et al.,
// "Edge-Avoiding À-Trous Wavelet Transform for fast Global Illumination Filtering", HPG 2010).  A post-pass over the
// float4 accumulator every render entry produces; no render kernel is involved.  sm_100a only.
#include "rt_kernels.cuh"
#include "rt_shade.cuh"

namespace rtd {

// --------------------------------------------------------------- feature pass ----
// One thread per pixel averages K camera samples (indices sample_offset .. sample_offset + K - 1): the primary rays the
// render traced for those samples (same Philox keys), their closest hit, the hit surface and one shade_terms() step with
// rp.flags cleared by the host entry.  Plane 0 (features[pixel]): mean outward normal and mean hit distance t*|d| over the
// samples that hit; plane 1 (features[npix + pixel]): mean albedo over all K samples and the fraction that hit.
// Albedo: scatter()'s attenuation (lambertian texture, metal / dielectric tint), E - bloom for an emitter, the world
// colour for a miss.  Single roundings are written out so that the oracle's restatement reproduces every value.
__global__ void __launch_bounds__(256) k_features(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp,
                                                  int use_bvh, int feature_spp, float4* __restrict__ features) {
    extern __shared__ __align__(16) uint32_t smem[];
    perlin_stage(smem, threadIdx.x, blockDim.x);
    __syncthreads();
    PerlinTab pt{smem, threadIdx.x & 31u};
    const uint32_t npix = uint32_t(rp.width) * uint32_t(rp.height);
    const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
    if (pixel >= npix) return;
    float nx = 0.f, ny = 0.f, nz = 0.f, dist = 0.f, ar = 0.f, ag = 0.f, ab = 0.f;
    int hits = 0;
    for (int k = 0; k < feature_spp; ++k) {
        const uint32_t sample = uint32_t(rp.sample_offset + k);
        const RayQ q = make_rayq(camera_ray(sc, rp, pixel, sample));
        const Hit h = closest_hit(sc, q, rp.tmin, use_bvh != 0);
        if (h.prim == RT_INVALID_ID) {
            ar = __fadd_rn(ar, rp.world_r);
            ag = __fadd_rn(ag, rp.world_g);
            ab = __fadd_rn(ab, rp.world_b);
            continue;
        }
        V3 p, n;
        hit_surface(sc, q, h, p, n);
        V3 E, att, direct = mk(0.f, 0.f, 0.f);
        Ray next;
        bool nee_vertex;
        uint32_t shadow_rays = 0;
        shade_terms(sc, rp, pt, q, h, pixel, sample, 1u, E, att, next, direct, nee_vertex, shadow_rays);
        if (load_mat(sc, __ldg(&sc.sph_c[h.prim]).y).kind == RT_MAT_EMITTER) // (shade_terms leaves att = 0 there)
            att = mk(__fsub_rn(E.x, rp.bloom), __fsub_rn(E.y, rp.bloom), __fsub_rn(E.z, rp.bloom));
        ++hits;
        nx = __fadd_rn(nx, n.x);
        ny = __fadd_rn(ny, n.y);
        nz = __fadd_rn(nz, n.z);
        const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(q.d.x, q.d.x), __fmul_rn(q.d.y, q.d.y)), __fmul_rn(q.d.z, q.d.z)));
        dist = __fadd_rn(dist, __fmul_rn(h.t, len));
        ar = __fadd_rn(ar, att.x);
        ag = __fadd_rn(ag, att.y);
        ab = __fadd_rn(ab, att.z);
    }
    const float fh = float(hits), fk = float(feature_spp);
    float4 f0 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (hits > 0) f0 = make_float4(__fdiv_rn(nx, fh), __fdiv_rn(ny, fh), __fdiv_rn(nz, fh), __fdiv_rn(dist, fh));
    features[pixel] = f0;
    features[size_t(npix) + pixel] = make_float4(__fdiv_rn(ar, fk), __fdiv_rn(ag, fk), __fdiv_rn(ab, fk), __fdiv_rn(fh, fk));
}

void launch_features(const DScene& sc, const DRenderParams& rp, bool use_bvh, int feature_spp, float4* features, cudaStream_t st) {
    const uint32_t npix = uint32_t(rp.width) * uint32_t(rp.height);
    if (npix == 0) return;
    const size_t smem = RT_PERLIN_SMEM_WORDS * sizeof(uint32_t);
    k_features<<<(npix + 255u) / 256u, 256, smem, st>>>(sc, rp, use_bvh ? 1 : 0, feature_spp, features);
}

// --------------------------------------------------------------- à-trous level ----
// Level i: 5x5 B3-spline taps h = (1, 4, 6, 4, 1)/16 per axis, 2^i pixels apart; taps outside the frame and neighbours
// without samples (w = 0) are skipped.  Tap weight
//   h * exp(-|c_p - c_q|^2 / (sigma_c 2^-i)^2 - |n_p - n_q|^2 / sigma_n^2 - |z_p - z_q| / (sigma_z max(z_p, z_q, eps))
//           - (|a_p - a_q|^2 + (f_p - f_q)^2) / sigma_a^2)
// with one __expf per tap, normalised by the sum of the weights.  Input colour: FROM_ACCUM = the render's accumulator,
// c = saturate(sum * rn(1 / count)); otherwise a previous level's output, whose valid pixels hold (c, 1).  A pixel without
// samples copies its input, so after the last level it still holds the accumulator's value and finalises exactly as
// rt_tonemap_device finalises it.
#define RT_ATROUS_EPS 1e-4f
struct AtrousLevel {
    int step;                            // 2^i
    float k_c, k_n, k_z, k_a;            // 1 / (sigma_c 2^-i)^2, 1 / sigma_n^2, 1 / sigma_z, 1 / sigma_a^2
};

template <bool FROM_ACCUM>
RT_DEV float3 mean_colour(float4 a) {
    if (!FROM_ACCUM) return make_float3(a.x, a.y, a.z);
    const float inv = __frcp_rn(a.w);
    return make_float3(__saturatef(__fmul_rn(a.x, inv)), __saturatef(__fmul_rn(a.y, inv)), __saturatef(__fmul_rn(a.z, inv)));
}

template <bool FROM_ACCUM>
__global__ void __launch_bounds__(256) k_atrous(const float4* __restrict__ in, const float4* __restrict__ features, int width,
                                                int height, const __grid_constant__ AtrousLevel lv, float4* __restrict__ out) {
    const int x = int(blockIdx.x * blockDim.x + threadIdx.x), y = int(blockIdx.y * blockDim.y + threadIdx.y);
    if (x >= width || y >= height) return;
    const size_t npix = size_t(width) * size_t(height), idx = size_t(y) * size_t(width) + size_t(x);
    const float4 a = __ldg(&in[idx]);
    if (!(a.w > 0.f)) {
        out[idx] = a;
        return;
    }
    const float3 c = mean_colour<FROM_ACCUM>(a);
    const float4 g0 = __ldg(&features[idx]), g1 = __ldg(&features[npix + idx]);
    const float h[5] = {1.f / 16.f, 4.f / 16.f, 6.f / 16.f, 4.f / 16.f, 1.f / 16.f};
    float sw = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int yy = y + dy * lv.step;
        if (yy < 0 || yy >= height) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int xx = x + dx * lv.step;
            if (xx < 0 || xx >= width) continue;
            const size_t q = size_t(yy) * size_t(width) + size_t(xx);
            const float4 b = __ldg(&in[q]);
            if (!(b.w > 0.f)) continue;
            const float3 cq = mean_colour<FROM_ACCUM>(b);
            const float4 q0 = __ldg(&features[q]), q1 = __ldg(&features[npix + q]);
            const float dr = c.x - cq.x, dg = c.y - cq.y, db = c.z - cq.z;
            const float ex = g0.x - q0.x, ey = g0.y - q0.y, ez = g0.z - q0.z;
            const float ar = g1.x - q1.x, ag = g1.y - q1.y, ab = g1.z - q1.z, af = g1.w - q1.w;
            const float zmax = fmaxf(fmaxf(g0.w, q0.w), RT_ATROUS_EPS);
            const float e = (dr * dr + dg * dg + db * db) * lv.k_c + (ex * ex + ey * ey + ez * ez) * lv.k_n +
                            __fdividef(fabsf(g0.w - q0.w), zmax) * lv.k_z + (ar * ar + ag * ag + ab * ab + af * af) * lv.k_a;
            const float w = h[dy + 2] * h[dx + 2] * __expf(-e);
            sw += w;
            sr += w * cq.x;
            sg += w * cq.y;
            sb += w * cq.z;
        }
    }
    const float inv = 1.f / sw; // > 0: the centre tap has weight (6/16)^2
    out[idx] = make_float4(sr * inv, sg * inv, sb * inv, 1.f);
}

void launch_atrous(const float4* in, bool from_accum, const float4* features, int width, int height, int level, float sigma_color,
                   float sigma_normal, float sigma_depth, float sigma_albedo, float4* out, cudaStream_t st) {
    if (width <= 0 || height <= 0) return;
    AtrousLevel lv;
    lv.step = 1 << level;
    const float sc = sigma_color / float(lv.step);
    lv.k_c = 1.f / (sc * sc);
    lv.k_n = 1.f / (sigma_normal * sigma_normal);
    lv.k_z = 1.f / sigma_depth;
    lv.k_a = 1.f / (sigma_albedo * sigma_albedo);
    const dim3 block(32, 8), grid(unsigned((width + 31) / 32), unsigned((height + 7) / 8));
    if (from_accum)
        k_atrous<true><<<grid, block, 0, st>>>(in, features, width, height, lv, out);
    else
        k_atrous<false><<<grid, block, 0, st>>>(in, features, width, height, lv, out);
}

} // namespace rtd
