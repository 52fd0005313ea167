// rt_shade.cuh — camera rays, textures (incl. Perlin), materials and the per-hit
// integrator step.  Semantics follow SURVEY.md §8a / §8a' item by item; every function
// cites the reference lines it restates.
#pragma once

#include "rt_intersect.cuh"

namespace rtd {

// ------------------------------------------------------------------ Perlin ----
// perlin_noise() / perlin_turbulence() are out-of-line functions and the octave loop is not unrolled: the shade kernels
// stay at ~3 800 SASS instructions (62 KB instead of 144 KB), which removed the instruction-cache stalls of the first
// version and lets ptxas fit 32 warps per SM (64 registers).
//
// Round 2 rewrote the lattice walk and the gradient for instruction count (ncu, C1: Perlin was 36 % of all executed
// warp instructions at 194 per octave, 108 of them the eight gradient selections, and the ALU pipe — selects, compares,
// logic — was the busiest pipe of the kernel; profiles/r02_c1_instruction_diet.md):
//  * ONE shared-memory table of 512 slots (the reference's doubled p[512], perlin_noise.h:43, so no index is ever
//    masked after the first).  Slot i = (p[i] * 8) | code(p[i]) << 16 | code(p[i + 1]) << 24: the low half is the BYTE
//    OFFSET of slot p[i] (slots are 8 bytes apart: two replicas, lane parity picks one), so the next level's address is
//    one add — `LDS.U16 [slot]` and `LDS.U16 [slot + 8]` fetch p[i] and p[i + 1] without any shift or mask —, and the two
//    high bytes are the gradient codes of the lattice points z and z + 1 in the form R2P turns into five predicates
//    with one instruction (bit 0: u = y, 1: v = y, 2: v = x, 3: negate u, 4: negate v; perlin_noise::grad,
//    perlin_noise.h:173-181).  A gradient is then R2P + 5 FSEL + FADD = 7 instructions instead of 13-14.
//  * per octave: 10 LDS + 7 address adds instead of 7 LDS + 33 shifts/masks/adds; 124 instead of 194 instructions.
// The arithmetic (operands, order, roundings) is unchanged: every value is bit-identical to the round-1 code.
// Ken Perlin's 2002 permutation (perlin_noise.h:24-37).  p[512] of the reference is
// this table twice (perlin_noise.h:43), so p[i] == perm[i & 255] for every index used.
__device__ const uint8_t k_perlin_perm[256] = {
    151, 160, 137, 91,  90,  15,  131, 13,  201, 95,  96,  53,  194, 233, 7,   225, 140, 36,  103, 30,  69,  142,
    8,   99,  37,  240, 21,  10,  23,  190, 6,   148, 247, 120, 234, 75,  0,   26,  197, 62,  94,  252, 219, 203,
    117, 35,  11,  32,  57,  177, 33,  88,  237, 149, 56,  87,  174, 20,  125, 136, 171, 168, 68,  175, 74,  165,
    71,  134, 139, 48,  27,  166, 77,  146, 158, 231, 83,  111, 229, 122, 60,  211, 133, 230, 220, 105, 92,  41,
    55,  46,  245, 40,  244, 102, 143, 54,  65,  25,  63,  161, 1,   216, 80,  73,  209, 76,  132, 187, 208, 89,
    18,  169, 200, 196, 135, 130, 116, 188, 159, 86,  164, 100, 109, 198, 173, 186, 3,   64,  52,  217, 226, 250,
    124, 123, 5,   202, 38,  147, 118, 126, 255, 82,  85,  212, 207, 206, 59,  227, 47,  16,  58,  17,  182, 189,
    28,  42,  223, 183, 170, 213, 119, 248, 152, 2,   44,  154, 163, 70,  221, 153, 101, 155, 167, 43,  172, 9,
    129, 22,  39,  253, 19,  98,  108, 110, 79,  113, 224, 232, 178, 185, 112, 104, 218, 246, 97,  228, 251, 34,
    242, 193, 238, 210, 144, 12,  191, 179, 162, 241, 81,  51,  145, 235, 249, 14,  239, 107, 49,  192, 214, 31,
    181, 199, 106, 157, 184, 84,  204, 176, 115, 121, 50,  45,  127, 4,   150, 254, 138, 236, 205, 93,  222, 114,
    67,  29,  24,  72,  243, 141, 128, 195, 78,  66,  215, 61,  156, 180};

#define RT_PERLIN_SLOTS 512u
#define RT_PERLIN_SMEM_WORDS (RT_PERLIN_SLOTS * 2u) // two replicas per slot: 4 KB per CTA
struct PerlinTab {
    const uint32_t* s; // shared memory, RT_PERLIN_SMEM_WORDS words
    uint32_t lane;
};
// gradient code of hash h (perlin_noise::grad, perlin_noise.h:173-181): u = h < 8 ? x : y;
// v = h < 4 ? y : (h == 12 || h == 14 ? x : z); result = (h & 1 ? -u : u) + (h & 2 ? -v : v)
RT_DEV uint32_t perlin_code(uint32_t hash) {
    const uint32_t h = hash & 15u;
    return (h >= 8u ? 1u : 0u) | (h < 4u ? 2u : 0u) | ((h == 12u || h == 14u) ? 4u : 0u) | ((h & 1u) << 3) | ((h & 2u) << 3);
}
RT_DEV void perlin_stage(uint32_t* smem, uint32_t tid, uint32_t nthreads) {
    for (uint32_t w = tid; w < RT_PERLIN_SMEM_WORDS; w += nthreads) {
        const uint32_t i = w >> 1;
        const uint32_t p0 = k_perlin_perm[i & 255u], p1 = k_perlin_perm[(i + 1u) & 255u];
        smem[w] = (p0 * 8u) | (perlin_code(p0) << 16) | (perlin_code(p1) << 24);
    }
}
// byte address of slot 0 of this lane's replica
RT_DEV const char* perlin_base(const PerlinTab& pt) { return reinterpret_cast<const char*>(pt.s) + ((pt.lane & 1u) << 2); }
// (p[i] * 8, p[i + 1] * 8) of the slot at byte address `slot`
RT_DEV uint32_t perlin_next(const char* slot) { return *reinterpret_cast<const uint16_t*>(slot); }
RT_DEV uint32_t perlin_next1(const char* slot) { return *reinterpret_cast<const uint16_t*>(slot + 8); }

// perlin_noise::grad (perlin_noise.h:173-181) from the code byte BYTE (2: lattice point z, 3: z + 1) of a slot word
template <int BYTE>
RT_DEV float perlin_grad(uint32_t w, float x, float y, float z) {
    constexpr int SH = 8 * BYTE;
    const bool uy = (w >> SH) & 1u, vy = (w >> (SH + 1)) & 1u, vx = (w >> (SH + 2)) & 1u, nu = (w >> (SH + 3)) & 1u, nv = (w >> (SH + 4)) & 1u;
    float u = uy ? y : x;
    float v = vx ? x : z;
    v = vy ? y : v;
    u = nu ? -u : u;
    v = nv ? -v : v;
    return u + v;
}
RT_DEV float perlin_ease(float t) { return t * t * t * (t * (t * 6.f - 15.f) + 10.f); } // :156-165
RT_DEV float perlin_lerp(float t, float a, float b) { return a + t * (b - a); }         // :167-171

// perlin_noise::noise (perlin_noise.h:46-105); `base` = perlin_base(pt)
RT_DEV float perlin_noise_body(const char* base, V3 p) {
    float fx = floorf(p.x), fy = floorf(p.y), fz = floorf(p.z);
    uint32_t xi = uint32_t(int(fx)) & 255u, yi = uint32_t(int(fy)) & 255u, zi = uint32_t(int(fz)) & 255u;
    float xf = p.x - fx, yf = p.y - fy, zf = p.z - fz;
    float u = perlin_ease(xf), v = perlin_ease(yf), w = perlin_ease(zf);
    const char* sx = base + xi * 8u;                    // slot xi
    const char* by = base + yi * 8u;                    // slot p[.] + yi  =  by + p[.] * 8
    const char* bz = base + zi * 8u;
    const char* sA = by + perlin_next(sx);              // slot A  = p[xi] + yi          (:67)
    const char* sB = by + perlin_next1(sx);             // slot B  = p[xi + 1] + yi      (:70)
    const uint32_t gaa = *reinterpret_cast<const uint32_t*>(bz + perlin_next(sA));  // slot AA = p[A] + zi: codes of p[AA], p[AA + 1]
    const uint32_t gab = *reinterpret_cast<const uint32_t*>(bz + perlin_next1(sA)); // slot AB = p[A + 1] + zi
    const uint32_t gba = *reinterpret_cast<const uint32_t*>(bz + perlin_next(sB));  // slot BA = p[B] + zi
    const uint32_t gbb = *reinterpret_cast<const uint32_t*>(bz + perlin_next1(sB)); // slot BB = p[B + 1] + zi
    float x1 = xf - 1.f, y1 = yf - 1.f, z1 = zf - 1.f;
    float res = perlin_lerp(
        w,
        perlin_lerp(v, perlin_lerp(u, perlin_grad<2>(gaa, xf, yf, zf), perlin_grad<2>(gba, x1, yf, zf)),
                    perlin_lerp(u, perlin_grad<2>(gab, xf, y1, zf), perlin_grad<2>(gbb, x1, y1, zf))),
        perlin_lerp(v, perlin_lerp(u, perlin_grad<3>(gaa, xf, yf, z1), perlin_grad<3>(gba, x1, yf, z1)),
                    perlin_lerp(u, perlin_grad<3>(gab, xf, y1, z1), perlin_grad<3>(gbb, x1, y1, z1))));
    return (res + 1.0f) / 2.0f;
}
static __device__ __noinline__ float perlin_noise(const PerlinTab& pt, V3 p) { return perlin_noise_body(perlin_base(pt), p); }

// perlin_noise::turbulance_noise, implementation 3 (perlin_noise.h:142-153), defaults
// lacunacity 2, gain .5, 6 octaves (perlin_noise.h:13-17).  ONE out-of-line call per 6-octave evaluation with the
// noise body inlined in its loop.
static __device__ __noinline__ float perlin_turbulence(const PerlinTab& pt, V3 p) {
    const char* base = perlin_base(pt);
    float frequency = 1.f, sum = 0.f, amplitude = 1.f;
#pragma unroll 1
    for (int i = 0; i < 6; ++i) {
        float r = perlin_noise_body(base, p * frequency);
        sum += fabsf(r * 2.f - 1.f) * amplitude;
        frequency *= 2.f;
        amplitude *= 0.5f;
    }
    return sum;
}

// ------------------------------------------------------------------ textures ----
RT_DEV DTexture load_tex(const DScene& sc, int32_t ix) {
    const float4* tp = reinterpret_cast<const float4*>(sc.texs + ix);
    float4 a = __ldg(tp), b = __ldg(tp + 1), c = __ldg(tp + 2);
    DTexture t;
    t.kind = __float_as_uint(a.x);
    t.even = __float_as_int(a.y);
    t.odd = __float_as_int(a.z);
    t.image = __float_as_int(a.w);
    t.c1x = b.x; t.c1y = b.y; t.c1z = b.z; t.density = b.w;
    t.c2x = c.x; t.c2y = c.y; t.c2z = c.z; t.hardness = c.w;
    return t;
}

// checker_texture::value (texture.h:41-48) only selects a child from p; children may be
// checkers themselves.  Returns the index of the leaf texture and loads it into `t`.  rt_scene_create refuses chains
// deeper than RT_MAX_CHECKER_DEPTH and cycles, so the loop always ends on a leaf.
RT_DEV int32_t resolve_texture(const DScene& sc, int32_t ix, V3 p, DTexture& t) {
    t = load_tex(sc, ix);
    for (int guard = 0; guard < RT_MAX_CHECKER_DEPTH && t.kind == RT_TEX_CHECKER; ++guard) {
        float sines = __sinf(10 * p.x) * __sinf(10 * p.y) * __sinf(10 * p.z);
        ix = sines < 0.f ? t.odd : t.even;
        t = load_tex(sc, ix);
    }
    return ix;
}

RT_DEV V3 tex_constant(const DTexture& t) { return mk(t.c1x, t.c1y, t.c1z); } // texture.h:22-24
RT_DEV V3 tex_perlin(const PerlinTab& pt, const DTexture& t, V3 p) {         // texture.h:58-59
    float v = perlin_noise(pt, p * t.density);
    return mk(v, v, v);
}
RT_DEV V3 tex_turbulence(const PerlinTab& pt, const DTexture& t, V3 p) { // texture.h:60-63: vec3(1) * 0.5 * turb(p * density)
    float v = __fmul_rz(0.5f, perlin_turbulence(pt, p * t.density));
    return mk(v, v, v);
}
RT_DEV V3 tex_marble(const PerlinTab& pt, const DTexture& t, V3 p) { // texture.h:65-75: turbulence of the UNSCALED p
    float value = 0.5f * (1 + __sinf((p.z * t.density + 7 * perlin_turbulence(pt, p))));
    V3 color1 = mk(0.925f, 0.816f, 0.78f);
    V3 color2 = mk(float(0.349 / 2), float(0.431 / 2), float(0.498 / 2));
    return color1 * value + color2 * (1 - value);
}
RT_DEV V3 tex_wood(const PerlinTab& pt, const DTexture& t, V3 p) { // texture.h:99-104
    float nn = t.hardness * perlin_noise(pt, p / t.density);
    nn -= floorf(nn);
    return (mk(t.c1x, t.c1y, t.c1z) * nn) + (mk(t.c2x, t.c2y, t.c2z) * (1.f - nn));
}
RT_DEV V3 tex_image(const DScene& sc, const DTexture& t, V3 n) { // image_texture::value (texture.h:118-132)
    float u, v;
    sphere_uv(n, u, v);
    const DImage& im = sc.images[t.image];
    int i = u * im.width;
    int j = (1 - v) * im.height - 0.001;
    if (i < 0) i = 0;
    if (j < 0) j = 0;
    if (i > im.width - 1) i = im.width - 1;
    if (j > im.height - 1) j = im.height - 1;
    float4 c = tex2D<float4>(im.tex, i + 0.5f, j + 0.5f); // nearest texel, row 0 = top
    return mk(c.x, c.y, c.z);
}

// text::value(u, v, p) of a non-checker texture.  (u,v) are only needed by image textures
// and are derived from the outward normal there (sphere.h:123-128).
RT_DEV V3 texture_leaf_value(const DScene& sc, const PerlinTab& pt, const DTexture& t, V3 n, V3 p) {
    switch (t.kind) {
    case RT_TEX_CONSTANT: return tex_constant(t);
    case RT_TEX_NOISE_PERLIN: return tex_perlin(pt, t, p);
    case RT_TEX_NOISE_TURBULANCE: return tex_turbulence(pt, t, p);
    case RT_TEX_NOISE_MARBLE: return tex_marble(pt, t, p);
    case RT_TEX_WOOD: return tex_wood(pt, t, p);
    case RT_TEX_IMAGE: return tex_image(sc, t, n);
    default: return mk(1.f, 1.f, 1.f);
    }
}

RT_DEV V3 texture_value(const DScene& sc, const PerlinTab& pt, int32_t ix, V3 n, V3 p) {
    DTexture t;
    resolve_texture(sc, ix, p, t);
    return texture_leaf_value(sc, pt, t, n, p);
}

// ------------------------------------------------------------------ camera ----
// render()'s per-sample set-up (main.cu:116-118) + camera::get_ray (camera.h:33-38).
// Draw order of the reference: jitter x, jitter y, lens disk, shutter time.
RT_DEV Ray camera_ray_of(const DCamera& cam, const DRenderParams& rp, uint32_t pixel, uint32_t sample) {
    const uint32_t j = fastdiv(pixel, rp.div_width), i = pixel - j * uint32_t(rp.width);
    U4 r0 = rng_block(rp.seed, pixel, sample, 0, 0);
    float s = float(i + u01(r0.x)) / float(rp.width);
    float t = float(j + u01(r0.y)) / float(rp.height);
    float dx, dy;
    sample_unit_disk(u01(r0.z), u01(r0.w), dx, dy);
    V3 rd = cam.lens_radius * mk(dx, dy, 0.f);
    V3 offset = cam.u * rd.x + cam.v * rd.y;
    float time = cam.t0;
    if (cam.t1 != cam.t0) {
        U4 r1 = rng_block(rp.seed, pixel, sample, 0, 1);
        time = __fadd_rn(cam.t0, __fmul_rn(u01(r1.x), __fsub_rn(cam.t1, cam.t0))); // single roundings: the same shutter time in every kernel
    }
    Ray r;
    r.o = cam.origin + offset;
    r.d = cam.lower_left + s * cam.horizontal + t * cam.vertical - cam.origin - offset;
    r.time = time;
    return r;
}

// The camera ray of a path: through the scene's camera, or in FRAMES instantiations through the camera of the sample's frame
template <int RM = RM_PLAIN>
RT_DEV Ray camera_ray(const DScene& sc, const DRenderParams& rp, uint32_t pixel, uint32_t sample) {
    if constexpr (RM == RM_FRAMES) {
        DCamera cam;
        const float* src = reinterpret_cast<const float*>(rp.frame_cams + frame_of(rp, sample));
        float* dst = reinterpret_cast<float*>(&cam);
#pragma unroll
        for (int k = 0; k < int(sizeof(DCamera) / sizeof(float)); ++k) dst[k] = __ldg(src + k);
        return camera_ray_of(cam, rp, pixel, sample);
    } else {
        return camera_ray_of(sc.cam, rp, pixel, sample);
    }
}

// ------------------------------------------------------------------ materials ----
RT_DEV DMaterial load_mat(const DScene& sc, uint32_t ix) {
    const float4* mp = reinterpret_cast<const float4*>(sc.mats + ix);
    float4 a = __ldg(mp), b = __ldg(mp + 1);
    DMaterial m;
    m.kind = __float_as_uint(a.x);
    m.tex = __float_as_int(a.y);
    m.ax = a.z; m.ay = a.w; m.az = b.x; m.param = b.y;
    m.pad0 = m.pad1 = 0.f;
    return m;
}

RT_DEV V3 reflect(V3 v, V3 n) { return v - 2.f * dot(v, n) * n; } // utils.h:93-97

// utils::refract (utils.h:107-122)
RT_DEV bool refract(V3 v, V3 n, float mu, V3& refracted) {
    V3 i = normalize(v);
    float in = dot(i, n);
    // Written with explicit single roundings: left to the compiler, `1 - in * in` was fused into an FMA in some kernels
    // and not in others (same source, different inlining context), and the refracted rays of the persistent-lane kernel
    // left the megakernel's by an ulp — 3.8 % of the pixels of the million-sphere frame (round-1 debugging run).
    float delta = __fsub_rn(1.f, __fmul_rn(__fmul_rn(mu, mu), __fsub_rn(1.f, __fmul_rn(in, in))));
    if (delta > 0) {
        refracted = mu * (i - n * in) - n * sqrtf(delta);
        return true;
    }
    return false;
}

// utils::shlick (utils.h:124-137)
RT_DEV float shlick(float cosine, float ref_id) {
    float r0 = div_rz((1.f - ref_id), (1.f + ref_id));
    r0 = __fmul_rz(r0, r0);
    return r0 + __fmul_rz((1.f - r0), __powf(1.f - cosine, 5.f));
}

// lambertian::scatter (material.h:105-116): target = p + n + ball; ray keeps rin's time
RT_DEV void scatter_lambertian(const RayQ& q, V3 p, V3 n, U4 r, Ray& out) {
    V3 target = p + n + sample_unit_ball(u01(r.x), u01(r.y), u01(r.z));
    out.o = p;
    out.d = target - p;
    out.time = q.time;
}

// ---- emitter importance sampling (RT_RENDER_EMITTER_SAMPLING; the reference README's roadmap item, README.md:27-28) ----
// In color() (main.cu:39-57) a path that reaches an emitter is worth emit + bloom, whatever it did before.  At a
// lambertian hit the reference draws d = n + uniform-in-ball (material.h:112), whose direction density about the
// normal is p_ref(w) = 2 cos^3(theta) / pi (the chord of the unit ball centred at n along w is 2 cos(theta); |d|
// along it has a density proportional to t^2).  The value of the vertex splits into
//     V = Int p_ref [next hit is a listed emitter] (emit + bloom)  +  Int p_ref [anything else] (rest of color())
// With the flag on, the first integral is estimated by ONE extra "shadow/emission" ray per lambertian hit, aimed
// uniformly into the cone of an emitter sphere chosen by solid angle (|d| from the reference's conditional law given w,
// 2 cos(theta) cbrt(u): tmin is in units of |d|), worth (p_ref / p_sel) (emit + bloom) if its closest hit is an
// emitter; the second by the reference's own scattered ray, which now counts 0 when its next hit is a listed
// emitter.  Same expectation, weights p_ref / p_sel of the order of an emitter's solid angle — never above the
// reference estimator's own range.  Ordinary colour-math FP32; nothing here is compared bit for bit.
struct LightCone {
    V3 axis;             // unit vector from p to the emitter's centre
    float one_minus_cos; // w is inside the cone  <=>  1 - dot(w, axis) <= one_minus_cos   (2 = every direction)
};
RT_DEV LightCone light_cone(const DScene& sc, uint32_t k, V3 p, float time) {
    const uint32_t prim = sc.lights[k];
    const float4 a = __ldg(&sc.sph_a[prim]);
    V3 c = mk(a.x, a.y, a.z);
    if (prim >= sc.n_static) c = moving_center(a, __ldg(&sc.sph_b[prim]), __uint_as_float(__ldg(&sc.sph_c[prim]).x), time);
    const float lx = c.x - p.x, ly = c.y - p.y, lz = c.z - p.z;
    const float d2 = lx * lx + ly * ly + lz * lz, r2 = a.w * a.w;
    LightCone lc;
    if (!(d2 > r2)) { // on or inside the emitter: every direction reaches it
        lc.axis = mk(0.f, 0.f, 1.f);
        lc.one_minus_cos = 2.f;
    } else {
        const float inv = 1.f / sqrtf(d2);
        lc.axis = V3{lx * inv, ly * inv, lz * inv};
        const float s2 = r2 / d2; // sin^2 of the half angle
        lc.one_minus_cos = fmaxf(s2 / (1.f + sqrtf(1.f - s2)), 1e-12f);
    }
    return lc;
}
// Is `prim` one of the emitter spheres the shadow rays sample?  (All of them unless the scene has more than RT_MAX_LIGHTS.)
RT_DEV bool light_listed(const DScene& sc, uint32_t prim) {
    bool listed = false;
    for (uint32_t k = 0; k < sc.n_lights; ++k) listed = listed || sc.lights[k] == prim;
    return listed;
}
// The shadow ray's direction `d` (with the reference's |d| law) at a lambertian hit (p, n); `rl` = Philox block (bounce, 2).
// Emitter k is chosen with probability proportional to its solid angle, the direction uniformly inside its cone, so
// p_sel(w) = (number of cones holding w) / (total solid angle) and p_ref / p_sel <= p_ref x total solid angle.
// Returns p_ref / p_sel, or 0 when the direction leaves below the horizon (p_ref = 0 there: no ray is traced).
RT_DEV float sample_light_direction(const DScene& sc, V3 p, V3 n, float time, U4 rl, V3& d) {
    const float inv_n = 1.f / sqrtf(n.x * n.x + n.y * n.y + n.z * n.z);
    float total = 0.f; // sum of (1 - cos half-angle) = total solid angle / 2 pi
    for (uint32_t j = 0; j < sc.n_lights; ++j) total += light_cone(sc, j, p, time).one_minus_cos;
    const float pick = u01(rl.x) * total;
    LightCone lc = light_cone(sc, 0u, p, time);
    uint32_t k = 0;
    float below = 0.f;
    for (uint32_t j = 0; j + 1u < sc.n_lights && !(pick <= below + lc.one_minus_cos); ++j) { // walk the cumulative sum
        below += lc.one_minus_cos;
        k = j + 1u;
        lc = light_cone(sc, k, p, time);
    }
    const float cz = 1.f - u01(rl.y) * lc.one_minus_cos; // cos of the angle to the axis, uniform over the cap
    const float sz = sqrtf(fmaxf(0.f, 1.f - cz * cz));
    float sn, cs;
    __sincosf(6.283185307179586f * u01(rl.z), &sn, &cs);
    const V3 ax = lc.axis; // orthonormal basis around it (Duff et al. 2017)
    const float sg = ax.z >= 0.f ? 1.f : -1.f;
    const float ka = -1.f / (sg + ax.z), kb = ax.x * ax.y * ka;
    const V3 t1 = V3{1.f + sg * ax.x * ax.x * ka, sg * kb, -sg * ax.x};
    const V3 t2 = V3{kb, sg + ax.y * ax.y * ka, -ax.y};
    const float e1 = sz * cs, e2 = sz * sn;
    const V3 w = V3{e1 * t1.x + e2 * t2.x + cz * ax.x, e1 * t1.y + e2 * t2.y + cz * ax.y, e1 * t1.z + e2 * t2.z + cz * ax.z};
    const float cos_t = (w.x * n.x + w.y * n.y + w.z * n.z) * inv_n;
    if (!(cos_t > 0.f)) return 0.f;
    const float len = 2.f * cos_t * fminf(cbrtf(u01(rl.w)), 0.99999994f);
    d = V3{w.x * len, w.y * len, w.z * len};
    const float p_ref = 0.6366197723675814f * cos_t * cos_t * cos_t; // 2 cos^3 / pi
    float holding = 0.f; // cones that hold w (the chosen one does by construction)
    for (uint32_t j = 0; j < sc.n_lights; ++j) {
        const LightCone lj = light_cone(sc, j, p, time);
        const float off = 1.f - (w.x * lj.axis.x + w.y * lj.axis.y + w.z * lj.axis.z);
        if (j == k || lj.one_minus_cos >= 2.f || off <= lj.one_minus_cos) holding += 1.f;
    }
    return p_ref * 6.283185307179586f * total / holding;
}
// The shadow/emission ray of one lambertian hit: (p_ref / p_sel) (emit + bloom) if its closest hit is a listed emitter.
RT_DEV V3 emitter_sample(const DScene& sc, const DRenderParams& rp, const PerlinTab& pt, V3 p, V3 n, float time, uint32_t pixel,
                         uint32_t sample, uint32_t bounce, uint32_t& rays) {
    V3 d;
    const float w = sample_light_direction(sc, p, n, time, rng_block(rp.seed, pixel, sample, bounce, 2), d);
    if (w == 0.f) return mk(0.f, 0.f, 0.f);
    Ray r;
    r.o = p;
    r.d = d;
    r.time = time;
    const RayQ q = make_rayq(r);
    const Hit h = closest_hit(sc, q, rp.tmin, true);
    ++rays;
    if (h.prim == RT_INVALID_ID) return mk(0.f, 0.f, 0.f);
    const DMaterial m = load_mat(sc, __ldg(&sc.sph_c[h.prim]).y);
    if (m.kind != RT_MAT_EMITTER || !light_listed(sc, h.prim)) return mk(0.f, 0.f, 0.f);
    V3 hp, hn;
    hit_surface(sc, q, h, hp, hn);
    const V3 e = texture_value(sc, pt, m.tex, hn, hp) * m.param + mk(rp.bloom, rp.bloom, rp.bloom); // emitter::emit + bloom
    return V3{e.x * w, e.y * w, e.z * w};
}
RT_DEV bool is_listed_emitter(const DScene& sc, uint32_t prim) {
    const float4 m0 = __ldg(reinterpret_cast<const float4*>(sc.mats + __ldg(&sc.sph_c[prim]).y));
    return __float_as_uint(m0.x) == RT_MAT_EMITTER && light_listed(sc, prim);
}

// metal::scatter (material.h:118-131): draws the ball sample even at roughness 0, ray time
// resets to 0 (ray.h:12 default), absorbed when dot(out, n) <= 0
RT_DEV bool scatter_metal(const RayQ& q, V3 p, V3 n, float roughness, U4 r, Ray& out) {
    V3 reflection = reflect(normalize(q.d), n);
    out.o = p;
    out.d = reflection + roughness * sample_unit_ball(u01(r.x), u01(r.y), u01(r.z));
    out.time = 0.f;
    return dot(out.d, n) > 0.f;
}

// dielectric::scatter (material.h:133-184); ray time resets to 0
RT_DEV void scatter_dielectric(const RayQ& q, V3 p, V3 n, float ri, U4 r, Ray& out) {
    V3 refraction_normal;
    V3 reflected = reflect(q.d, n);
    float mu, cosine;
    float ddn = dot(q.d, n);
    if (ddn > 0.f) {
        refraction_normal = -n;
        mu = ri;
        cosine = __fdiv_rn(ddn, length(q.d));
        cosine = sqrt_rz(__fsub_rn(1.f, __fmul_rn(__fmul_rn(ri, ri), __fsub_rn(1.f, __fmul_rn(cosine, cosine))))); // no contraction, as above
    } else {
        refraction_normal = n;
        mu = 1.f / ri;
        cosine = __fdiv_rn(-ddn, length(q.d));
    }
    float reflect_prob;
    V3 refracted = mk(0.f, 0.f, 0.f);
    if (refract(q.d, refraction_normal, mu, refracted)) {
        reflect_prob = shlick(cosine, ri);
    } else {
        reflect_prob = 1.f;
    }
    out.o = p;
    out.d = (u01(r.w) < reflect_prob) ? reflected : refracted;
    out.time = 0.f;
}

// The terms of one integrator step at an accepted hit — the body of color()'s loop (main.cu:45-55):
//   E = m.emit(h) + bloom;  `att`/`out` = what m.scatter(...) produces.  Returns false when scatter() does
// (emitter, absorbed metal ray): the path's value is then E.  `bounce` counts from 1 for the RNG key.
// RT_RENDER_EMITTER_SAMPLING: a lambertian hit also traces its shadow/emission ray — `direct` receives that ray's
// contribution, `rays` counts it, and `nee_vertex` tells the caller that a listed emitter hit by `out` is worth 0.
RT_DEV bool shade_terms(const DScene& sc, const DRenderParams& rp, const PerlinTab& pt, const RayQ& q, Hit h,
                        uint32_t pixel, uint32_t sample, uint32_t bounce, V3& E, V3& att, Ray& out, V3& direct, bool& nee_vertex,
                        uint32_t& rays) {
    V3 p, n;
    hit_surface(sc, q, h, p, n);
    DMaterial m = load_mat(sc, __ldg(&sc.sph_c[h.prim]).y);
    V3 bloom = mk(rp.bloom, rp.bloom, rp.bloom);
    att = mk(0.f, 0.f, 0.f);
    nee_vertex = false;
    if (m.kind == RT_MAT_EMITTER) { // emitter::emit / scatter (material.h:42-52)
        E = texture_value(sc, pt, m.tex, n, p) * m.param + bloom;
        return false;
    }
    E = mk(0.f, 0.f, 0.f) + bloom; // material::emit (material.h:14-16)
    U4 r = rng_block(rp.seed, pixel, sample, bounce, 0);
    if (m.kind == RT_MAT_LAMBERTIAN) {
        scatter_lambertian(q, p, n, r, out);
        att = texture_value(sc, pt, m.tex, n, p);
        // (the reference traces at most max_depth rays per path, main.cu:42: the shadow ray stands for trace bounce + 1)
        if ((rp.flags & RT_RENDER_EMITTER_SAMPLING) && sc.n_lights > 0u && int(bounce) < rp.max_depth) {
            const V3 c = emitter_sample(sc, rp, pt, p, n, q.time, pixel, sample, bounce, rays);
            direct = V3{direct.x + c.x, direct.y + c.y, direct.z + c.z};
            nee_vertex = true;
        }
        return true;
    }
    att = mk(m.ax, m.ay, m.az);
    if (m.kind == RT_MAT_METAL) return scatter_metal(q, p, n, m.param, r, out); // false: absorbed, the value is E
    scatter_dielectric(q, p, n, m.param, r, out);
    return true;
}

// A <- E + att*A (main.cu:51) or A <- E when the path ends.  Returns true if the path continues.
RT_DEV bool shade_hit(const DScene& sc, const DRenderParams& rp, const PerlinTab& pt, const RayQ& q, Hit h,
                      uint32_t pixel, uint32_t sample, uint32_t bounce, V3& A, Ray& out, V3& direct, bool& nee_vertex, uint32_t& rays) {
    V3 E, att;
    if (!shade_terms(sc, rp, pt, q, h, pixel, sample, bounce, E, att, out, direct, nee_vertex, rays)) {
        A = E;
        return false;
    }
    A = E + att * A;
    return true;
}

} // namespace rtd
