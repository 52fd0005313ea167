// rt_jpeg_decode.cu — device half of the JPEG reader (image-texture ingest, SURVEY.md §8f-2): from the quantised DCT
// coefficients the host half decoded (rt_jpeg_decode_host.cpp) to the float image stbi_loadf returns (main.cu:376-380).
// Every stage is stb_image v2.26's INTEGER arithmetic (its SSE2 kernels are written to be bit-identical to the scalar
// code they replace, stb_image.h:2450-2452,3556-3557), so the result equals stb's byte for byte:
//   k_jpegd_idct   one thread per 8x8 block: coefficient * quantiser (16-bit wrap, stb:2998-3003,2164), the two passes of
//                  the jidctint-derived IDCT with its 12-bit constants and roundings (stb:2358-2447) -> u8 plane
//   k_jpegd_rgb    one thread per output pixel: each component's sample through the up-sampling filter stb picks from
//                  its sampling factors (stb:3355-3426,3545-3555; which source rows a picture row blends is stb's
//                  line0/line1 state machine, stb:3828-3841, replayed on the host into two small row tables),
//                  then the fixed-point YCbCr -> RGB of stb:3558-3583 and byte / 255.f (stb:1797-1810)
// Bound: HBM (2 B/coefficient read, 1 B/sample written and read, 12 B/pixel written); sized for scene-load time, not
// for the frame loop.
#include <vector>

#include "rt_jpeg_decode.cuh"
#include "rt_kernels.cuh"

namespace rtd {

namespace {

#define F2F(x) ((int)(((x) * 4096 + 0.5)))
#define FSH(x) ((x) * 4096)
// one 1-D pass of stb's IDCT (STBI__IDCT_1D, stb:2358-2395)
#define IDCT_1D(s0, s1, s2, s3, s4, s5, s6, s7)  \
    int t0, t1, t2, t3, p1, p2, p3, p4, p5, x0, x1, x2, x3; \
    p2 = s2;                                     \
    p3 = s6;                                     \
    p1 = (p2 + p3) * F2F(0.5411961f);            \
    t2 = p1 + p3 * F2F(-1.847759065f);           \
    t3 = p1 + p2 * F2F(0.765366865f);            \
    p2 = s0;                                     \
    p3 = s4;                                     \
    t0 = FSH(p2 + p3);                           \
    t1 = FSH(p2 - p3);                           \
    x0 = t0 + t3;                                \
    x3 = t0 - t3;                                \
    x1 = t1 + t2;                                \
    x2 = t1 - t2;                                \
    t0 = s7;                                     \
    t1 = s5;                                     \
    t2 = s3;                                     \
    t3 = s1;                                     \
    p3 = t0 + t2;                                \
    p4 = t1 + t3;                                \
    p1 = t0 + t3;                                \
    p2 = t1 + t2;                                \
    p5 = (p3 + p4) * F2F(1.175875602f);          \
    t0 = t0 * F2F(0.298631336f);                 \
    t1 = t1 * F2F(2.053119869f);                 \
    t2 = t2 * F2F(3.072711026f);                 \
    t3 = t3 * F2F(1.501321110f);                 \
    p1 = p5 + p1 * F2F(-0.899976223f);           \
    p2 = p5 + p2 * F2F(-2.562915447f);           \
    p3 = p3 * F2F(-1.961570560f);                \
    p4 = p4 * F2F(-0.390180644f);                \
    t3 += p1 + p4;                               \
    t2 += p2 + p3;                               \
    t1 += p2 + p4;                               \
    t0 += p1 + p3;

__device__ __forceinline__ uint8_t clamp8(int x) { return uint8_t(x < 0 ? 0 : (x > 255 ? 255 : x)); }

struct DequantTab {
    uint16_t q[64];
};

__global__ void __launch_bounds__(128)
    k_jpegd_idct(const int16_t* __restrict__ coeff, const __grid_constant__ DequantTab dq, int blocks_w, int used_w, int used_h, int w2,
                 uint8_t* __restrict__ plane) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= used_w * used_h) return;
    const int bx = b % used_w, by = b / used_w;
    const int16_t* c = coeff + size_t(by * blocks_w + bx) * 64;
    int d[64], val[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) d[i] = int(int16_t(int(c[i]) * int(dq.q[i]))); // data[i] *= dequant[i] in 16 bits
    // columns (stb:2404-2428; its all-zero shortcut gives the same values as the general path)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        IDCT_1D(d[i], d[8 + i], d[16 + i], d[24 + i], d[32 + i], d[40 + i], d[48 + i], d[56 + i])
        x0 += 512;
        x1 += 512;
        x2 += 512;
        x3 += 512;
        val[i] = (x0 + t3) >> 10;
        val[56 + i] = (x0 - t3) >> 10;
        val[8 + i] = (x1 + t2) >> 10;
        val[48 + i] = (x1 - t2) >> 10;
        val[16 + i] = (x2 + t1) >> 10;
        val[40 + i] = (x2 - t1) >> 10;
        val[24 + i] = (x3 + t0) >> 10;
        val[32 + i] = (x3 - t0) >> 10;
    }
    // rows (stb:2430-2447): remove the 2^17 scale, round, re-centre on 128, clamp
    uint8_t* o = plane + size_t(by * 8) * w2 + bx * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i, o += w2) {
        const int* v = val + 8 * i;
        IDCT_1D(v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7])
        x0 += 65536 + (128 << 17);
        x1 += 65536 + (128 << 17);
        x2 += 65536 + (128 << 17);
        x3 += 65536 + (128 << 17);
        uint8_t r[8];
        r[0] = clamp8((x0 + t3) >> 17);
        r[7] = clamp8((x0 - t3) >> 17);
        r[1] = clamp8((x1 + t2) >> 17);
        r[6] = clamp8((x1 - t2) >> 17);
        r[2] = clamp8((x2 + t1) >> 17);
        r[5] = clamp8((x2 - t1) >> 17);
        r[3] = clamp8((x3 + t0) >> 17);
        r[4] = clamp8((x3 - t0) >> 17);
        *reinterpret_cast<uint2*>(o) = make_uint2(r[0] | r[1] << 8 | r[2] << 16 | r[3] << 24, r[4] | r[5] << 8 | r[6] << 16 | r[7] << 24);
    }
}

enum { RS_COPY = 0, RS_V2, RS_H2, RS_HV2, RS_GENERIC };

struct PlaneView {
    const uint8_t* plane;
    const int* near_row; // [height] source row blended with weight 3 (or copied)
    const int* far_row;  // [height]
    int w2, w_lores, hs, kind;
};
struct RgbParams {
    PlaneView c[3];
    int width, height, n_comp, is_rgb;
};

// sample of one component at picture position (x, y): stb's resample_row_* (stb:3355-3426, 3545-3555) evaluated at x
__device__ __forceinline__ int upsample(const PlaneView& p, int x, int y) {
    const uint8_t* nr = p.plane + size_t(p.near_row[y]) * p.w2;
    const uint8_t* fr = p.plane + size_t(p.far_row[y]) * p.w2;
    const int w = p.w_lores;
    switch (p.kind) {
    case RS_COPY: return nr[x];
    case RS_V2: return (3 * nr[x] + fr[x] + 2) >> 2;
    case RS_H2: {
        if (w == 1) return nr[0];
        const int i = x >> 1;
        if (x == 0) return nr[0];
        if (x == 2 * w - 1) return nr[w - 1];
        if (x == 2 * (w - 1)) return (nr[w - 2] * 3 + nr[w - 1] + 2) >> 2; // stb's last even sample weights the PREVIOUS input
        return (x & 1) ? (3 * nr[i] + nr[i + 1] + 2) >> 2 : (3 * nr[i] + nr[i - 1] + 2) >> 2;
    }
    case RS_HV2: {
        if (w == 1) return (3 * nr[0] + fr[0] + 2) >> 2;
        if (x == 0) return (3 * nr[0] + fr[0] + 2) >> 2;
        if (x == 2 * w - 1) return (3 * nr[w - 1] + fr[w - 1] + 2) >> 2;
        const int i = (x + 1) >> 1; // x = 2i-1 or 2i
        const int ta = 3 * nr[i - 1] + fr[i - 1], tb = 3 * nr[i] + fr[i];
        return (x & 1) ? (3 * ta + tb + 8) >> 4 : (3 * tb + ta + 8) >> 4;
    }
    default: return nr[x / p.hs];
    }
}

#define F2FIX(x) (((int)((x) * 4096.0f + 0.5f)) << 8)
__global__ void __launch_bounds__(256) k_jpegd_rgb(const __grid_constant__ RgbParams P, float* __restrict__ out) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(P.width) * P.height) return;
    const int x = int(i % P.width), y = int(i / P.width);
    const int s0 = upsample(P.c[0], x, y) & 255;
    if (P.n_comp == 1) {
        out[i] = float(s0) / 255.0f;
        return;
    }
    const int s1 = upsample(P.c[1], x, y) & 255, s2 = upsample(P.c[2], x, y) & 255;
    int r, g, b;
    if (P.is_rgb) {
        r = s0;
        g = s1;
        b = s2;
    } else { // stbi__YCbCr_to_RGB_row (stb:3558-3583)
        const int y_fixed = (s0 << 20) + (1 << 19);
        const int cr = s2 - 128, cb = s1 - 128;
        r = y_fixed + cr * F2FIX(1.40200f);
        g = y_fixed + (cr * -F2FIX(0.71414f)) + ((cb * -F2FIX(0.34414f)) & 0xffff0000);
        b = y_fixed + cb * F2FIX(1.77200f);
        r >>= 20;
        g >>= 20;
        b >>= 20;
        r = r < 0 ? 0 : (r > 255 ? 255 : r);
        g = g < 0 ? 0 : (g > 255 ? 255 : g);
        b = b < 0 ? 0 : (b > 255 ? 255 : b);
    }
    out[3 * i + 0] = float(r) / 255.0f;
    out[3 * i + 1] = float(g) / 255.0f;
    out[3 * i + 2] = float(b) / 255.0f;
}

} // namespace

// which source rows a picture row uses: stb's per-component line0/line1/ystep state machine (stb:3800-3841)
void jpeg_row_tables(const rtj::CoefficientImage& img, int k, std::vector<int>& near_row, std::vector<int>& far_row) {
    const rtj::Component& c = img.comp[k];
    const int vs = img.v_max / c.v;
    int ystep = vs >> 1, ypos = 0, line0 = 0, line1 = 0;
    near_row.resize(img.height);
    far_row.resize(img.height);
    for (int j = 0; j < img.height; ++j) {
        const bool y_bot = ystep >= (vs >> 1);
        near_row[j] = y_bot ? line1 : line0;
        far_row[j] = y_bot ? line0 : line1;
        if (++ystep >= vs) {
            ystep = 0;
            line0 = line1;
            if (++ypos < c.y) line1 += 1;
        }
    }
}

int jpeg_resample_kind(int hs, int vs) {
    if (hs == 1 && vs == 1) return RS_COPY;
    if (hs == 1 && vs == 2) return RS_V2;
    if (hs == 2 && vs == 1) return RS_H2;
    if (hs == 2 && vs == 2) return RS_HV2;
    return RS_GENERIC;
}

cudaError_t jpeg_pixels_device(const rtj::CoefficientImage& img, float* out_dev, cudaStream_t st, float* ms_device) {
    TimingEvent ev[2];
    RTD_TRY(ev[0].create());
    RTD_TRY(ev[1].create());
    RgbParams P{};
    P.width = img.width;
    P.height = img.height;
    P.n_comp = img.n_comp;
    P.is_rgb = img.is_rgb ? 1 : 0;
    std::vector<std::vector<int>> rows(2 * img.n_comp);
    struct Planes {
        PoolBuffer<int16_t> coeff;
        PoolBuffer<uint8_t> plane;
        PoolBuffer<int> near_rows, far_rows;
    };
    std::vector<Planes> owned(img.n_comp); // the device copies of each component
    RTD_TRY(cudaEventRecord(ev[0].ev, st));
    for (int k = 0; k < img.n_comp; ++k) {
        const rtj::Component& c = img.comp[k];
        Planes& o = owned[k];
        RTD_TRY(o.coeff.alloc(c.coeff.size(), st));
        RTD_TRY(o.plane.alloc(size_t(c.w2) * c.h2, st));
        RTD_TRY(o.near_rows.alloc(size_t(img.height), st));
        RTD_TRY(o.far_rows.alloc(size_t(img.height), st));
        RTD_TRY(cudaMemcpyAsync(o.coeff.get(), c.coeff.data(), c.coeff.size() * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        jpeg_row_tables(img, k, rows[2 * k], rows[2 * k + 1]);
        RTD_TRY(cudaMemcpyAsync(o.near_rows.get(), rows[2 * k].data(), size_t(img.height) * sizeof(int), cudaMemcpyHostToDevice, st));
        RTD_TRY(cudaMemcpyAsync(o.far_rows.get(), rows[2 * k + 1].data(), size_t(img.height) * sizeof(int), cudaMemcpyHostToDevice, st));
        DequantTab dq;
        for (int i = 0; i < 64; ++i) dq.q[i] = img.dequant[c.tq][i];
        const int used_w = (c.x + 7) >> 3, used_h = (c.y + 7) >> 3; // the blocks stb transforms (stb:3012-3019)
        k_jpegd_idct<<<(used_w * used_h + 127) / 128, 128, 0, st>>>(o.coeff.get(), dq, c.blocks_w, used_w, used_h, c.w2, o.plane.get());
        const int hs = img.h_max / c.h, vs = img.v_max / c.v;
        P.c[k] = PlaneView{o.plane.get(), o.near_rows.get(), o.far_rows.get(), c.w2, (img.width + hs - 1) / hs, hs, jpeg_resample_kind(hs, vs)};
    }
    const size_t npix = size_t(img.width) * img.height;
    k_jpegd_rgb<<<unsigned((npix + 255) / 256), 256, 0, st>>>(P, out_dev);
    RTD_TRY(cudaGetLastError());
    RTD_TRY(cudaEventRecord(ev[1].ev, st));
    RTD_TRY(cudaStreamSynchronize(st)); // the host vectors above are pageable staging buffers
    if (ms_device) RTD_TRY(cudaEventElapsedTime(ms_device, ev[0].ev, ev[1].ev));
    return cudaSuccess;
}

} // namespace rtd
