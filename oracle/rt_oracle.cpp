// oracle/rt_oracle.cpp — TEST INFRASTRUCTURE.  CPU restatement of the per-pixel render path of
// slimem/raytracing_renderer_cuda, function by function, each citing the reference lines it
// follows.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
// legs may load this; the product (librt_b200.so) never does and has no CPU fallback.
//
// PARITY PIN: with sampler 0 / arith 0 this file reproduces oracle/_ref/libref_cpu.so — the
// reference's own headers compiled for the host through oracle/shim — bit for bit: closest
// hits, unit functions and whole renders (tests/test_oracle_pin.py; golden copies of those
// outputs are committed under tests/golden/ for machines without /root/reference).  With
// arith 1 the closest-hit arithmetic follows the contraction pattern of the reference's sm_100
// SASS and reproduces the reference GPU kernel's (id, t, p, n) bit for bit
// (tests/golden/ref_gpu_trace_*.npz, recorded from oracle/_ref/ref_harness on a B200).
// Whole frames of config C1 are also held against the reference's own committed output, renders/earth_emitter.jpg
// (as its 4x4 box filter, tests/golden/ref_render_earth_emitter_300x150.png): 36.9 dB at 64 spp, 44.4 dB at
// 1200x600x25 spp, noise-limited (tests/test_reference_render_fixture.py).
//
// Two axes select what is being restated:
//   arith   0  host arithmetic: every vec3 op is a true round-toward-zero op (rz_math.h), scalar
//              glue is round-to-nearest, nothing is fused (g++ -ffp-contract=off)
//           1  as 0, but sphere::hit's `dot(oc,oc) - r*r` and `b*b - a*c` are fused the way
//              ptxas fuses them in the reference kernel (FFMA, see csrc/rt_intersect.cuh)
//   sampler 0  the reference's sampling: one sequential generator per pixel, rejection sampling
//              of the unit ball / disk (utils.h:61-91), draw order of main.cu:116-118
//           1  the product's sampling: Philox4x32-10 keyed on (pixel, sample, bounce), direct
//              (non-rejection) sampling of the same distributions — what csrc/rt_device.cuh does
//
// NOT PINNED (nothing in the reference to pin against): rt_render_params.flags & RT_RENDER_EMITTER_SAMPLING, sampler 1
// only — the restatement of the product's shadow-ray estimator (the reference README names emitter sampling as future
// work, README.md:27-28).  It is checked by properties (tests/test_emitter_sampling.py); with flags == 0, which is what
// every parity test uses, none of that code runs.
#include "rt_oracle.h"

#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "oracle_rng.h"
#include "rz_math.h"

namespace {

// ------------------------------------------------------------------ vec3 (vec3.h) ----
struct V3 {
    float x, y, z;
};
inline V3 mk(float x, float y, float z) { return V3{x, y, z}; }
inline V3 operator+(V3 a, V3 b) { return mk(rz::add(a.x, b.x), rz::add(a.y, b.y), rz::add(a.z, b.z)); }   // vec3.h:258-269
inline V3 operator-(V3 a, V3 b) { return mk(rz::sub(a.x, b.x), rz::sub(a.y, b.y), rz::sub(a.z, b.z)); }   // vec3.h:270-281
inline V3 operator*(V3 a, V3 b) { return mk(rz::mul(a.x, b.x), rz::mul(a.y, b.y), rz::mul(a.z, b.z)); }   // vec3.h:282-293
inline V3 operator*(V3 a, float t) { return mk(rz::mul(a.x, t), rz::mul(a.y, t), rz::mul(a.z, t)); }      // vec3.h:318-329
inline V3 operator*(float t, V3 a) { return a * t; }                                                      // vec3.h:306-317
inline V3 operator/(V3 a, float t) { return mk(rz::div(a.x, t), rz::div(a.y, t), rz::div(a.z, t)); }      // vec3.h:330-341
inline V3 operator-(V3 a) { return mk(-a.x, -a.y, -a.z); }
// vec3::dot / sq_length (vec3.h:168-179,208-219): truncated products, round-to-nearest sums
inline float dot(V3 a, V3 b) { return (rz::mul(a.x, b.x) + rz::mul(a.y, b.y)) + rz::mul(a.z, b.z); }
inline float length(V3 a) { return rz::sqrt(dot(a, a)); } // vec3.h:153-166
inline V3 normalize(V3 a) {                               // vec3.h:199-205
    if (a.x == 0.f && a.y == 0.f && a.z == 0.f) return a;
    return a / length(a);
}
inline V3 cross(V3 a, V3 b) { // vec3.h:220-243
    return mk(rz::sub(rz::mul(a.y, b.z), rz::mul(a.z, b.y)), rz::mul(rz::sub(rz::mul(a.x, b.z), rz::mul(a.z, b.x)), -1.f),
              rz::sub(rz::mul(a.x, b.y), rz::mul(a.y, b.x)));
}

struct Ray {
    V3 o, d;
    float time;
};

// ------------------------------------------------------------------ scene ----
struct Camera { // camera.h:40-47
    V3 origin, lower_left, horizontal, vertical, u, v, w;
    float lens_radius, t0, t1;
};

} // namespace

struct orc_scene {
    std::vector<rt_sphere> spheres;
    std::vector<rt_material> materials;
    std::vector<rt_texture> textures;
    std::vector<std::vector<float>> images;
    std::vector<int32_t> image_wh;
    Camera cam;
    std::vector<uint32_t> lights; // emitter spheres in list order, at most RT_MAX_LIGHTS (RT_RENDER_EMITTER_SAMPLING)
};

namespace {

// camera ctor (camera.h:7-31).  __tanf becomes tanf on the host (as in the shim).
Camera make_camera(const rt_camera& c) {
    Camera k;
    k.t0 = c.time0;
    k.t1 = c.time1;
    k.lens_radius = rz::div(c.aperture, 2.f);
    float theta = float(double(c.vfov) * M_PI / double(180.f)); // `vfov * M_PI / 180.f` is evaluated in double
    float half_height = tanf(rz::div(theta, 2.f));
    float half_width = rz::mul(c.aspect, half_height);
    V3 lookfrom = mk(c.lookfrom[0], c.lookfrom[1], c.lookfrom[2]), lookat = mk(c.lookat[0], c.lookat[1], c.lookat[2]);
    V3 up = mk(c.up[0], c.up[1], c.up[2]);
    k.origin = lookfrom;
    k.w = normalize(lookfrom - lookat);
    k.u = normalize(cross(up, k.w));
    k.v = cross(k.w, k.u);
    // `half_width * focus_dist * _u`: float*float (round-to-nearest) first, then float*vec3
    k.lower_left = k.origin - (half_width * c.focus_dist) * k.u - (half_height * c.focus_dist) * k.v - c.focus_dist * k.w;
    k.horizontal = ((2 * half_width) * c.focus_dist) * k.u;
    k.vertical = ((2 * half_height) * c.focus_dist) * k.v;
    return k;
}

// ------------------------------------------------------------------ intersection ----
struct Hit {
    float t;
    uint32_t prim;
    V3 p, n;
    float u, v;
    bool uv_set;
};

// sphere::get_sphere_uv (sphere.h:61-83): atan2f/asinf in float, the affine maps in double
inline void sphere_uv(V3 n, float& u, float& v) {
    float phi = atan2f(n.z, n.x);
    float theta = asinf(n.y);
    u = float(1 - (phi + M_PI) / (2 * M_PI));
    v = float((theta + M_PI_2) / M_PI);
}

// moving_sphere::center (sphere.h:49-52)
inline V3 moving_center(const rt_sphere& s, float time) {
    V3 c0 = mk(s.center0[0], s.center0[1], s.center0[2]), c1 = mk(s.center1[0], s.center1[1], s.center1[2]);
    return c0 + ((time - s.time0) / (s.time1 - s.time0)) * (c1 - c0);
}

inline void quadratic(const Ray& r, V3 center, float radius, int arith, float& a, float& b, float& delta) {
    V3 oc = r.o - center;
    a = dot(r.d, r.d);
    b = dot(oc, r.d);
    if (arith == 1) { // the reference kernel's SASS: FFMA(-r, r, dot) and FFMA(b, b, -(a*c))
        float c = fmaf(-radius, radius, dot(oc, oc));
        delta = fmaf(b, b, -(a * c));
    } else {
        float c = dot(oc, oc) - radius * radius;
        delta = b * b - a * c;
    }
}

// sphere::hit (sphere.h:86-140): delta < 0 rejects; roots tested with inclusive bounds
bool sphere_hit(const rt_sphere& s, const Ray& r, float tmin, float tmax, int arith, Hit& h) {
    V3 c = mk(s.center0[0], s.center0[1], s.center0[2]);
    float a, b, delta;
    quadratic(r, c, s.radius, arith, a, b, delta);
    if (delta < 0) return false;
    float sq = sqrtf(delta);
    float root = (-b - sq) / a;
    if (root < tmin || root > tmax) {
        root = (-b + sq) / a;
        if (root < tmin || root > tmax) return false;
    }
    h.t = root;
    h.p = r.o + root * r.d; // ray::point_at_parameter (ray.h:28-30)
    h.n = (h.p - c) / s.radius;
    sphere_uv(h.n, h.u, h.v);
    h.uv_set = true;
    return true;
}

// moving_sphere::hit (sphere.h:157-190): delta > 0 strictly, bounds exclusive, u/v untouched
bool moving_sphere_hit(const rt_sphere& s, const Ray& r, float tmin, float tmax, int arith, Hit& h) {
    V3 c = moving_center(s, r.time);
    float a, b, delta;
    quadratic(r, c, s.radius, arith, a, b, delta);
    if (!(delta > 0)) return false;
    float sq = sqrtf(delta);
    float t = (-b - sq) / a;
    if (!(t < tmax && t > tmin)) {
        t = (-b + sq) / a;
        if (!(t < tmax && t > tmin)) return false;
    }
    h.t = t;
    h.p = r.o + t * r.d;
    h.n = (h.p - c) / s.radius;
    h.uv_set = false;
    return true;
}

// hitable_list::hit with no BVH (hitable_list.h:66-78): first-found wins ties.  The reference
// reuses one temporary record, so a moving sphere inherits the u/v of the last static candidate
// that was accepted before it (sphere.h:168-175 never writes them).
bool scene_hit(const orc_scene& sc, const Ray& r, float tmin, float tmax, int arith, Hit& out) {
    bool any = false;
    float closest = tmax;
    Hit tmp;
    tmp.u = tmp.v = 0.f;
    tmp.uv_set = false;
    for (uint32_t i = 0; i < sc.spheres.size(); ++i) {
        const rt_sphere& s = sc.spheres[i];
        bool ok = (s.flags & RT_SPHERE_MOVING) ? moving_sphere_hit(s, r, tmin, closest, arith, tmp)
                                               : sphere_hit(s, r, tmin, closest, arith, tmp);
        if (ok && tmp.t < closest) {
            any = true;
            closest = tmp.t;
            out = tmp;
            out.prim = i;
        }
    }
    return any;
}

// ------------------------------------------------------------------ Perlin (perlin_noise.h) ----
const uint8_t k_perm[256] = { // Ken Perlin's reference permutation (perlin_noise.h:24-37)
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
inline uint32_t P(uint32_t i) { return k_perm[i & 255u]; } // p[512] = the table twice (perlin_noise.h:41-44)

inline float grad(uint32_t hash, float x, float y, float z) { // perlin_noise.h:173-181
    uint32_t h = hash & 15u;
    float u = h < 8 ? x : y;
    float v = h < 4 ? y : (h == 12 || h == 14) ? x : z;
    return ((h & 1) == 0 ? u : -u) + ((h & 2) == 0 ? v : -v);
}
inline float ease(float t) { return t * t * t * (t * (t * 6 - 15) + 10); } // perlin_noise.h:156-165
inline float lerp(float t, float a, float b) { return a + t * (b - a); }   // perlin_noise.h:167-171

float perlin_noise(V3 pt) { // perlin_noise.h:46-105
    float xf = pt.x, yf = pt.y, zf = pt.z;
    uint32_t xi = uint32_t(int(floorf(pt.x))) & 255u, yi = uint32_t(int(floorf(pt.y))) & 255u,
             zi = uint32_t(int(floorf(pt.z))) & 255u;
    xf -= floorf(xf);
    yf -= floorf(yf);
    zf -= floorf(zf);
    float u = ease(xf), v = ease(yf), w = ease(zf);
    uint32_t A = P(xi) + yi, AA = P(A) + zi, AB = P(A + 1) + zi;
    uint32_t B = P(xi + 1) + yi, BA = P(B) + zi, BB = P(B + 1) + zi;
    float res = lerp(
        w,
        lerp(v, lerp(u, grad(P(AA), xf, yf, zf), grad(P(BA), xf - 1, yf, zf)),
             lerp(u, grad(P(AB), xf, yf - 1, zf), grad(P(BB), xf - 1, yf - 1, zf))),
        lerp(v, lerp(u, grad(P(AA + 1), xf, yf, zf - 1), grad(P(BA + 1), xf - 1, yf, zf - 1)),
             lerp(u, grad(P(AB + 1), xf, yf - 1, zf - 1), grad(P(BB + 1), xf - 1, yf - 1, zf - 1))));
    return (res + 1.0f) / 2.0f;
}

float turbulence(V3 p) { // perlin_noise.h:142-153, defaults lacunacity 2, gain .5, 6 octaves (:13-17)
    float frequency = 1.f, sum = 0.0f, amplitude = 1.f;
    for (int i = 0; i < 6; ++i) {
        float r = perlin_noise(p * frequency);
        sum += fabsf(r * 2 - 1) * amplitude;
        frequency *= 2.f;
        amplitude *= 0.5f;
    }
    return sum;
}

// ------------------------------------------------------------------ textures (texture.h) ----
V3 texture_value(const orc_scene& sc, int32_t ix, float u, float v, V3 p) {
    const rt_texture* t = &sc.textures[size_t(ix)];
    // checker_texture::value (texture.h:41-48), as far as the product resolves it: rt_scene_create refuses deeper chains and
    // cycles, so a description it accepts never reaches the guard
    for (int guard = 0; guard < RT_MAX_CHECKER_DEPTH && t->kind == RT_TEX_CHECKER; ++guard) {
        float sines = sinf(10 * p.x) * sinf(10 * p.y) * sinf(10 * p.z);
        t = &sc.textures[size_t(sines < 0.f ? t->odd : t->even)];
    }
    switch (t->kind) {
    case RT_TEX_CONSTANT: return mk(t->color1[0], t->color1[1], t->color1[2]); // texture.h:22-24
    case RT_TEX_NOISE_PERLIN: return mk(1, 1, 1) * perlin_noise(p * t->density); // texture.h:58-59
    case RT_TEX_NOISE_TURBULANCE: return (mk(1, 1, 1) * 0.5f) * turbulence(p * t->density); // texture.h:60-63
    case RT_TEX_NOISE_MARBLE: {                                                             // texture.h:65-75
        float value = 0.5f * (1 + sinf((p.z * t->density + 7 * turbulence(p))));
        V3 color1 = mk(float(0.925), float(0.816), float(0.78));
        V3 color2 = mk(float(0.349 / 2), float(0.431 / 2), float(0.498 / 2));
        return color1 * value + color2 * (1 - value);
    }
    case RT_TEX_WOOD: { // texture.h:99-104
        float n = t->hardness * perlin_noise(mk(p.x, p.y, p.z) / t->density);
        n -= floorf(n);
        return (mk(t->color1[0], t->color1[1], t->color1[2]) * n) + (mk(t->color2[0], t->color2[1], t->color2[2]) * (1.f - n));
    }
    case RT_TEX_IMAGE: { // image_texture::value (texture.h:118-132); int <- float, int <- double
        int W = sc.image_wh[2 * size_t(t->image)], H = sc.image_wh[2 * size_t(t->image) + 1];
        int i = int(u * W);
        int j = int((1 - v) * H - 0.001);
        if (i < 0) i = 0;
        if (j < 0) j = 0;
        if (i > W - 1) i = W - 1;
        if (j > H - 1) j = H - 1;
        const float* px = sc.images[size_t(t->image)].data() + (size_t(j) * W + i) * 3;
        return mk(px[0], px[1], px[2]);
    }
    default: return mk(1, 1, 1);
    }
}

// ------------------------------------------------------------------ optics (utils.h) ----
inline V3 reflect(V3 v, V3 n) { return v - (2.f * dot(v, n)) * n; } // utils.h:93-97: 2.f * float first, then * vec3

bool refract(V3 v, V3 n, float mu, V3& refracted) { // utils.h:107-122
    V3 i = normalize(v);
    float in = dot(i, n);
    float delta = 1.f - mu * mu * (1 - in * in);
    if (delta > 0) {
        refracted = mu * (i - n * in) - n * sqrtf(delta);
        return true;
    }
    return false;
}

float shlick(float cosine, float ri) { // utils.h:124-137 (device branch)
    float r0 = rz::div(1.f - ri, 1.f + ri);
    r0 = rz::mul(r0, r0);
    return r0 + rz::mul(1.f - r0, powf(1.f - cosine, 5.f));
}

// ------------------------------------------------------------------ samplers ----
struct Sampler {
    int mode; // 0 reference, 1 product
    orng_state seq;
    uint32_t seed, pixel, sample;
};

// Philox4x32-10, identical to csrc/rt_device.cuh
struct U4 {
    uint32_t x, y, z, w;
};
U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = uint64_t(0xD2511F53u) * c0, p1 = uint64_t(0xCD9E8D57u) * c2;
        uint32_t hi0 = uint32_t(p0 >> 32), lo0 = uint32_t(p0), hi1 = uint32_t(p1 >> 32), lo1 = uint32_t(p1);
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}
inline U4 rng_block(const Sampler& s, uint32_t bounce, uint32_t blk) {
    return philox4x32_10(s.pixel, s.sample, (bounce << 8) | blk, 0x52544232u, s.seed, 0x42323030u);
}
inline float u01(uint32_t x) { return fmaf(float(x), 2.3283064365386963e-10f, 1.1641532182693481e-10f); }

// utils::random_point_unit_sphere (utils.h:61-77).  g++ evaluates the three constructor
// arguments right to left, so the first draw lands in z (pinned against libref_cpu.so).
V3 ball_reference(orng_state* st) {
    V3 p;
    do {
        float c = orng_uniform(st), b = orng_uniform(st), a = orng_uniform(st);
        p = 2.f * mk(a, b, c) - mk(1.f, 1.f, 1.f);
    } while (dot(p, p) >= 1.f);
    return p;
}
V3 disk_reference(orng_state* st) { // utils.h:79-91
    V3 p;
    do {
        float b = orng_uniform(st), a = orng_uniform(st);
        p = 2.f * mk(a, b, 0) - mk(1.f, 1.f, 0.f);
    } while (dot(p, p) >= 1.f);
    return p;
}
// the product's direct samplers (csrc/rt_device.cuh: sample_unit_ball / sample_unit_disk)
V3 ball_product(float u1, float u2, float u3) {
    float z = fmaf(-2.f, u1, 1.f);
    float rxy = sqrtf(fmaxf(0.f, fmaf(-z, z, 1.f)));
    float ang = 6.283185307179586f * u2;
    float s = sinf(ang), c = cosf(ang);
    float rad = fminf(cbrtf(u3), 0.99999994f);
    return V3{rad * rxy * c, rad * rxy * s, rad * z};
}

// ------------------------------------------------------------------ camera::get_ray ----
Ray camera_ray(const orc_scene& sc, Sampler& sm, int i, int j, int width, int height) {
    const Camera& cam = sc.cam;
    float s, t, time;
    V3 rd;
    if (sm.mode == 0) { // main.cu:116-118 + camera.h:33-38, draw order: jitter x, jitter y, disk, time
        s = float(i + orng_uniform(&sm.seq)) / float(width);
        t = float(j + orng_uniform(&sm.seq)) / float(height);
        rd = cam.lens_radius * disk_reference(&sm.seq);
        time = cam.t0 + orng_uniform(&sm.seq) * (cam.t1 - cam.t0);
    } else { // csrc/rt_shade.cuh camera_ray
        U4 r0 = rng_block(sm, 0, 0);
        s = float(i + u01(r0.x)) / float(width);
        t = float(j + u01(r0.y)) / float(height);
        float rad = fminf(sqrtf(u01(r0.z)), 0.99999994f), ang = 6.283185307179586f * u01(r0.w);
        rd = cam.lens_radius * mk(rad * cosf(ang), rad * sinf(ang), 0.f);
        time = cam.t0;
        if (cam.t1 != cam.t0) time = cam.t0 + u01(rng_block(sm, 0, 1).x) * (cam.t1 - cam.t0);
    }
    V3 offset = cam.u * rd.x + cam.v * rd.y;
    Ray r;
    r.o = cam.origin + offset;
    r.d = cam.lower_left + s * cam.horizontal + t * cam.vertical - cam.origin - offset;
    r.time = time;
    return r;
}

// ------------------------------------------------------------------ emitter importance sampling ----
// Not in the reference (its README names it as future work, README.md:27-28): the restatement of the product's
// RT_RENDER_EMITTER_SAMPLING estimator (csrc/rt_shade.cuh; include/rt_api.h).  In color() a path that reaches an emitter
// is worth emit + bloom, whatever it did before (main.cu:49-55).  The reference's lambertian direction n + uniform-in-ball
// (material.h:112) has the direction density p_ref = 2 cos^3(theta) / pi, so the value of a lambertian hit splits into
//   Int p_ref [next hit is a listed emitter] (emit + bloom)  +  Int p_ref [anything else] (rest of color()).
// The first integral is estimated by one shadow/emission ray aimed uniformly into the cone of an emitter sphere
// chosen by solid angle (|d| from the reference's conditional law 2 cos(theta) cbrt(u)), worth (p_ref / p_sel)(emit + bloom)
// when its closest hit is a listed emitter; the second by the reference's scattered ray, which counts 0 when its next
// hit is a listed emitter.  Plain float arithmetic.
struct LightCone {
    V3 axis;
    float one_minus_cos;
};
LightCone light_cone(const orc_scene& sc, uint32_t k, V3 p, float time) {
    const rt_sphere& s = sc.spheres[sc.lights[k]];
    V3 c = (s.flags & RT_SPHERE_MOVING) ? moving_center(s, time) : mk(s.center0[0], s.center0[1], s.center0[2]);
    const float lx = c.x - p.x, ly = c.y - p.y, lz = c.z - p.z;
    const float d2 = lx * lx + ly * ly + lz * lz, r2 = s.radius * s.radius;
    LightCone lc;
    if (!(d2 > r2)) {
        lc.axis = mk(0.f, 0.f, 1.f);
        lc.one_minus_cos = 2.f;
    } else {
        const float inv = 1.f / sqrtf(d2);
        lc.axis = V3{lx * inv, ly * inv, lz * inv};
        const float s2 = r2 / d2;
        lc.one_minus_cos = fmaxf(s2 / (1.f + sqrtf(1.f - s2)), 1e-12f);
    }
    return lc;
}
bool is_listed_emitter(const orc_scene& sc, uint32_t prim) {
    for (uint32_t k : sc.lights)
        if (k == prim) return true; // the list holds emitter spheres only
    return false;
}
// returns p_ref / p_sel and the shadow ray's direction; 0 = below the horizon (p_ref = 0), no ray.  The emitter is
// chosen with probability proportional to its solid angle: p_sel = (cones holding w) / (total solid angle).
float sample_light_direction(const orc_scene& sc, V3 p, V3 n, float time, U4 rl, V3& d) {
    const uint32_t n_lights = uint32_t(sc.lights.size());
    const float inv_n = 1.f / sqrtf(n.x * n.x + n.y * n.y + n.z * n.z);
    float total = 0.f;
    for (uint32_t j = 0; j < n_lights; ++j) total += light_cone(sc, j, p, time).one_minus_cos;
    const float pick = u01(rl.x) * total;
    LightCone lc = light_cone(sc, 0u, p, time);
    uint32_t k = 0;
    float below = 0.f;
    for (uint32_t j = 0; j + 1u < n_lights && !(pick <= below + lc.one_minus_cos); ++j) {
        below += lc.one_minus_cos;
        k = j + 1u;
        lc = light_cone(sc, k, p, time);
    }
    const float cz = 1.f - u01(rl.y) * lc.one_minus_cos;
    const float sz = sqrtf(fmaxf(0.f, 1.f - cz * cz));
    const float ang = 6.283185307179586f * u01(rl.z);
    const float sn = sinf(ang), cs = cosf(ang);
    const V3 ax = lc.axis;
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
    const float p_ref = 0.6366197723675814f * cos_t * cos_t * cos_t;
    float holding = 0.f;
    for (uint32_t j = 0; j < n_lights; ++j) {
        const LightCone lj = light_cone(sc, j, p, time);
        const float off = 1.f - (w.x * lj.axis.x + w.y * lj.axis.y + w.z * lj.axis.z);
        if (j == k || lj.one_minus_cos >= 2.f || off <= lj.one_minus_cos) holding += 1.f;
    }
    return p_ref * 6.283185307179586f * total / holding;
}

// ------------------------------------------------------------------ materials (material.h) ----
// Returns false when the path ends at this hit (emitter, absorbed metal ray).
bool scatter(const orc_scene& sc, const rt_material& m, const Ray& rin, const Hit& h, Sampler& sm, uint32_t bounce,
             V3& attenuation, Ray& rout) {
    U4 rn{0, 0, 0, 0};
    if (sm.mode == 1 && m.kind != RT_MAT_EMITTER) rn = rng_block(sm, bounce, 0);
    switch (m.kind) {
    case RT_MAT_LAMBERTIAN: { // material.h:105-116
        V3 ball = sm.mode == 0 ? ball_reference(&sm.seq) : ball_product(u01(rn.x), u01(rn.y), u01(rn.z));
        V3 target = h.p + h.n + ball;
        rout = Ray{h.p, target - h.p, rin.time};
        attenuation = texture_value(sc, m.texture, h.u, h.v, h.p);
        return true;
    }
    case RT_MAT_METAL: { // material.h:118-131: the ball sample is drawn even at roughness 0; time resets to 0
        V3 reflection = reflect(normalize(rin.d), h.n);
        V3 ball = sm.mode == 0 ? ball_reference(&sm.seq) : ball_product(u01(rn.x), u01(rn.y), u01(rn.z));
        rout = Ray{h.p, reflection + m.param * ball, 0.f};
        attenuation = mk(m.albedo[0], m.albedo[1], m.albedo[2]);
        return dot(rout.d, h.n) > 0.f;
    }
    case RT_MAT_DIELECTRIC: { // material.h:133-184
        const float ri = m.param;
        V3 refraction_normal, reflected = reflect(rin.d, h.n);
        float mu, cosine;
        attenuation = mk(m.albedo[0], m.albedo[1], m.albedo[2]);
        if (dot(rin.d, h.n) > 0.f) {
            refraction_normal = -h.n;
            mu = ri;
            cosine = dot(rin.d, h.n) / length(rin.d);
            cosine = rz::sqrt(1.f - ri * ri * (1 - cosine * cosine));
        } else {
            refraction_normal = h.n;
            mu = 1.f / ri;
            cosine = -dot(rin.d, h.n) / length(rin.d);
        }
        float reflect_prob;
        V3 refracted = mk(0, 0, 0);
        if (refract(rin.d, refraction_normal, mu, refracted)) reflect_prob = shlick(cosine, ri);
        else reflect_prob = 1.f;
        float xi = sm.mode == 0 ? orng_uniform(&sm.seq) : u01(rn.w);
        rout = Ray{h.p, xi < reflect_prob ? reflected : refracted, 0.f};
        return true;
    }
    default: return false; // emitter::scatter (material.h:42-48)
    }
}

inline V3 emit(const orc_scene& sc, const rt_material& m, const Hit& h) {
    if (m.kind != RT_MAT_EMITTER) return mk(0.f, 0.f, 0.f);     // material::emit (material.h:14-16)
    return texture_value(sc, m.texture, h.u, h.v, h.p) * m.param; // emitter::emit (material.h:50-52)
}

// ------------------------------------------------------------------ color() (main.cu:35-74) ----
// The shadow/emission ray of a lambertian hit (RT_RENDER_EMITTER_SAMPLING, product sampler only).
V3 emitter_sample(const orc_scene& sc, const Hit& at, float time, Sampler& sm, uint32_t bounce, const rt_render_params& rp, int arith,
                  unsigned long long* rays) {
    V3 d;
    const float w = sample_light_direction(sc, at.p, at.n, time, rng_block(sm, bounce, 2), d);
    if (w == 0.f) return mk(0.f, 0.f, 0.f);
    Hit h;
    ++*rays;
    if (!scene_hit(sc, Ray{at.p, d, time}, rp.tmin, FLT_MAX, arith, h)) return mk(0.f, 0.f, 0.f);
    const rt_material& m = sc.materials[sc.spheres[h.prim].material];
    if (m.kind != RT_MAT_EMITTER || !is_listed_emitter(sc, h.prim)) return mk(0.f, 0.f, 0.f);
    if (!h.uv_set) sphere_uv(h.n, h.u, h.v);
    const V3 e = emit(sc, m, h) + mk(rp.bloom, rp.bloom, rp.bloom);
    return V3{e.x * w, e.y * w, e.z * w};
}

V3 color(const orc_scene& sc, Ray r, Sampler& sm, const rt_render_params& rp, int arith, unsigned long long* rays) {
    V3 A = mk(rp.world[0], rp.world[1], rp.world[2]);
    const V3 bloom = mk(rp.bloom, rp.bloom, rp.bloom);
    const bool nee = sm.mode == 1 && (rp.flags & RT_RENDER_EMITTER_SAMPLING) && !sc.lights.empty();
    V3 direct = mk(0.f, 0.f, 0.f); // shadow/emission rays of the path; x + 0.f is exact without the flag
    bool nee_vertex = false;       // `r` leaves a lambertian hit that traced its shadow ray
    auto total = [&direct](V3 v) { return V3{v.x + direct.x, v.y + direct.y, v.z + direct.z}; };
    for (int bounce = 1; bounce <= rp.max_depth; ++bounce) {
        Hit h;
        ++*rays;
        if (!scene_hit(sc, r, rp.tmin, FLT_MAX, arith, h)) return total(A);
        if (sm.mode == 1 && !h.uv_set) sphere_uv(h.n, h.u, h.v); // the product derives u/v from n for every sphere kind
        const rt_material& m = sc.materials[sc.spheres[h.prim].material];
        if (nee_vertex && m.kind == RT_MAT_EMITTER && is_listed_emitter(sc, h.prim)) return total(mk(0.f, 0.f, 0.f));
        Ray next;
        V3 att;
        V3 e = emit(sc, m, h) + bloom;
        if (!scatter(sc, m, r, h, sm, uint32_t(bounce), att, next)) return total(e);
        nee_vertex = false;
        if (nee && m.kind == RT_MAT_LAMBERTIAN && bounce < rp.max_depth) { // the shadow ray stands for trace bounce + 1
            const V3 c = emitter_sample(sc, h, r.time, sm, uint32_t(bounce), rp, arith, rays);
            direct = V3{direct.x + c.x, direct.y + c.y, direct.z + c.z};
            nee_vertex = true;
        }
        A = e + att * A;
        r = next;
    }
    return total(mk(0.f, 0.f, 0.f));
}

void store3(float* out, V3 v) {
    out[0] = v.x;
    out[1] = v.y;
    out[2] = v.z;
}

} // namespace

extern "C" {

orc_scene* orc_scene_create(const rt_scene_desc* d) {
    if (!d) return nullptr;
    orc_scene* s = new orc_scene();
    s->spheres.assign(d->spheres, d->spheres + d->n_spheres);
    s->materials.assign(d->materials, d->materials + d->n_materials);
    s->textures.assign(d->textures, d->textures + d->n_textures);
    for (uint32_t i = 0; i < d->n_images; ++i) {
        const rt_image& im = d->images[i];
        s->images.emplace_back(im.rgb, im.rgb + size_t(im.width) * im.height * 3);
        s->image_wh.push_back(im.width);
        s->image_wh.push_back(im.height);
    }
    s->cam = make_camera(d->camera);
    for (uint32_t i = 0; i < d->n_spheres && s->lights.size() < RT_MAX_LIGHTS; ++i)
        if (d->materials[d->spheres[i].material].kind == RT_MAT_EMITTER) s->lights.push_back(i);
    return s;
}

void orc_scene_destroy(orc_scene* s) { delete s; }

void orc_trace(const orc_scene* s, const rt_ray* rays, size_t n, float tmin, int arith, rt_hit* hits) {
    for (size_t i = 0; i < n; ++i) {
        const rt_ray& in = rays[i];
        Ray r{mk(in.origin[0], in.origin[1], in.origin[2]), mk(in.direction[0], in.direction[1], in.direction[2]), in.time};
        Hit h;
        rt_hit out;
        memset(&out, 0, sizeof out);
        if (scene_hit(*s, r, tmin, FLT_MAX, arith, h)) {
            out.t = h.t;
            out.id = s->spheres[h.prim].id;
            store3(out.p, h.p);
            store3(out.n, h.n);
            out.u = h.u;
            out.v = h.v;
        } else {
            out.t = FLT_MAX;
            out.id = RT_INVALID_ID;
        }
        hits[i] = out;
    }
}

// render (main.cu:97-132).  accum: W*H*4 floats (sum r, g, b, sample count), index j*W+i with
// j = 0 the bottom row — the layout of rt_render_accum.  Sampler 0 sums with vec3::operator+=
// (truncating adds, main.cu:119); sampler 1 sums in sample order with round-to-nearest adds.
void orc_render(const orc_scene* s, const rt_render_params* rp, int sampler, int arith, int nthreads, float* accum,
                unsigned long long* rays_out) {
    const int W = rp->width, H = rp->height;
    if (nthreads < 1) nthreads = 1;
    std::atomic<int> next_row{0};
    std::atomic<unsigned long long> total{0};
    auto work = [&]() {
        unsigned long long rays = 0;
        for (;;) {
            int j = next_row.fetch_add(1);
            if (j >= H) break;
            for (int i = 0; i < W; ++i) {
                size_t index = size_t(j) * size_t(W) + size_t(i);
                Sampler sm;
                sm.mode = sampler;
                sm.seed = rp->seed;
                sm.pixel = uint32_t(index);
                orng_init(rp->seed + index, 0, 0, &sm.seq); // init_rand_state (main.cu:91)
                V3 col = mk(0.f, 0.f, 0.f);
                for (int k = 0; k < rp->spp; ++k) {
                    sm.sample = uint32_t(k + rp->sample_offset);
                    Ray r = camera_ray(*s, sm, i, j, W, H);
                    V3 c = color(*s, r, sm, *rp, arith, &rays);
                    if (sampler == 0) col = col + c;
                    else col = mk(col.x + c.x, col.y + c.y, col.z + c.z);
                }
                accum[index * 4 + 0] = col.x;
                accum[index * 4 + 1] = col.y;
                accum[index * 4 + 2] = col.z;
                accum[index * 4 + 3] = float(rp->spp);
            }
        }
        total += rays;
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    if (rays_out) *rays_out = total.load();
}

// One integrator step per caller-supplied ray with the product's sampling (Philox key: pixel = ray index,
// sample 0, bounce 1): the counterpart of rt_shade_probe.
void orc_shade_probe(const orc_scene* s, const rt_ray* rays, size_t n, const rt_render_params* rp, int arith,
                     rt_shade_sample* out) {
    for (size_t i = 0; i < n; ++i) {
        const rt_ray& in = rays[i];
        Ray r{mk(in.origin[0], in.origin[1], in.origin[2]), mk(in.direction[0], in.direction[1], in.direction[2]), in.time};
        rt_shade_sample o;
        memset(&o, 0, sizeof o);
        o.id = RT_INVALID_ID;
        Hit h;
        if (scene_hit(*s, r, rp->tmin, FLT_MAX, arith, h)) {
            if (!h.uv_set) sphere_uv(h.n, h.u, h.v);
            const rt_material& m = s->materials[s->spheres[h.prim].material];
            Sampler sm;
            sm.mode = 1;
            sm.seed = rp->seed;
            sm.pixel = uint32_t(i);
            sm.sample = 0;
            Ray next{mk(0, 0, 0), mk(0, 0, 0), 0.f};
            V3 att = mk(0, 0, 0);
            V3 e = emit(*s, m, h) + mk(rp->bloom, rp->bloom, rp->bloom);
            bool cont = scatter(*s, m, r, h, sm, 1u, att, next);
            o.id = s->spheres[h.prim].id;
            o.continues = cont ? 1u : 0u;
            o.t = h.t;
            store3(o.emitted, e);
            if (m.kind != RT_MAT_EMITTER) store3(o.attenuation, att);
            if (cont) {
                store3(o.scattered.origin, next.o);
                store3(o.scattered.direction, next.d);
                o.scattered.time = next.time;
            }
        }
        out[i] = o;
    }
}

// Pixel finalisation (main.cu:124-127): col /= spp (vec3.h:138-151: rz(1/f), truncated
// multiplies), saturate, per-channel truncated sqrt.  accum as above; out: W*H*3.
void orc_tonemap(const float* accum, int width, int height, float* out_rgb) {
    for (size_t i = 0; i < size_t(width) * size_t(height); ++i) {
        float inv = rz::div(1.0f, accum[4 * i + 3]);
        for (int c = 0; c < 3; ++c) out_rgb[3 * i + c] = rz::sqrt(rz::saturate(rz::mul(accum[4 * i + c], inv)));
    }
}

float orc_perlin_noise(const float p[3]) { return perlin_noise(mk(p[0], p[1], p[2])); }
float orc_turbulence(const float p[3]) { return turbulence(mk(p[0], p[1], p[2])); }
void orc_texture_value(const orc_scene* s, int tex, float u, float v, const float p[3], float out[3]) {
    store3(out, texture_value(*s, tex, u, v, mk(p[0], p[1], p[2])));
}
void orc_reflect(const float v[3], const float n[3], float out[3]) {
    store3(out, reflect(mk(v[0], v[1], v[2]), mk(n[0], n[1], n[2])));
}
int orc_refract(const float v[3], const float n[3], float mu, float out[3]) {
    V3 r = mk(0, 0, 0);
    bool ok = refract(mk(v[0], v[1], v[2]), mk(n[0], n[1], n[2]), mu, r);
    store3(out, r);
    return ok ? 1 : 0;
}
float orc_shlick(float cosine, float ri) { return shlick(cosine, ri); }
void orc_sphere_uv(const float n[3], float* u, float* v) { sphere_uv(mk(n[0], n[1], n[2]), *u, *v); }
// The shadow ray of a lambertian hit at (p, n, time) with the Philox key (pixel = index, sample 0, bounce 1): direction
// and p_ref / p_sel (0: none).  Unit hook of the emitter-sampling tests.
float orc_light_sample(const orc_scene* s, const float p[3], const float n[3], float time, uint32_t seed, uint32_t index,
                       float dir[3]) {
    Sampler sm;
    sm.mode = 1;
    sm.seed = seed;
    sm.pixel = index;
    sm.sample = 0;
    V3 d = mk(0.f, 0.f, 0.f);
    const float w = sample_light_direction(*s, mk(p[0], p[1], p[2]), mk(n[0], n[1], n[2]), time, rng_block(sm, 1, 2), d);
    store3(dir, d);
    return w;
}
void orc_camera_ray(const orc_scene* s, float s_, float t_, unsigned long long seed, rt_ray* out) {
    // camera::get_ray (camera.h:33-38) with a caller-seeded sequential generator
    orng_state st;
    orng_init(seed, 0, 0, &st);
    const Camera& cam = s->cam;
    V3 rd = cam.lens_radius * disk_reference(&st);
    V3 offset = cam.u * rd.x + cam.v * rd.y;
    float time = cam.t0 + orng_uniform(&st) * (cam.t1 - cam.t0);
    V3 o = cam.origin + offset;
    V3 d = cam.lower_left + s_ * cam.horizontal + t_ * cam.vertical - cam.origin - offset;
    store3(out->origin, o);
    store3(out->direction, d);
    out->time = time;
}

} // extern "C"
