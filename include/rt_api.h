/*
 * rt_api.h — C-ABI of the B200-native path tracer (librt_b200.so).
 *
 * This is the drop-in boundary for the per-pixel render path of
 * slimem/raytracing_renderer_cuda (SURVEY.md §8b).  The reference has no FFI;
 * its "API" is (i) the device-side scene constructors called from
 * populate_scene_balls (src/main.cu:188-356) and (ii) the `render` kernel
 * launch + framebuffer convention (src/main.cu:97-132, :442-449, :475-491).
 * (i) becomes the flat POD scene description below (filled by the header-only
 * façade in include/rt/scene.hpp, which keeps the reference's class names and
 * constructor signatures); (ii) becomes rt_render*().
 *
 * Plain C: pointers and sizes only, no C++/torch types.  Every entry returns
 * an rt_status; the message of the last failure on the calling thread is
 * available from rt_last_error().  The library never calls exit() or
 * cudaDeviceReset() (reference: check_cuda, src/main.cu:23-30, does both).
 *
 * There is NO CPU fallback: every compute entry fails with RT_ERR_NO_DEVICE /
 * RT_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef RT_API_H
#define RT_API_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_API_VERSION 1
#define RT_INVALID_ID 0xFFFFFFFFu

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID_ARG = 1,
    RT_ERR_CUDA = 2,
    RT_ERR_OOM = 3,
    RT_ERR_UNSUPPORTED = 4,
    RT_ERR_NO_DEVICE = 5,
    RT_ERR_IO = 6
} rt_status;

/* ---- scene description (POD) ------------------------------------------- */

/* material kinds; reference classes in src/material.h */
enum {
    RT_MAT_LAMBERTIAN = 0, /* lambertian(const text*)            material.h:59-70,105-116 */
    RT_MAT_METAL = 1,      /* metal(vec3 albedo, float roughness) material.h:72-88,118-131 */
    RT_MAT_DIELECTRIC = 2, /* dielectric(float ri, vec3 tint)     material.h:90-103,133-184 */
    RT_MAT_EMITTER = 3     /* emitter(const text*, intensity=1)   material.h:38-56 (= diffuse_light) */
};

/* texture kinds; reference classes in src/texture.h */
enum {
    RT_TEX_CONSTANT = 0,   /* constant_texture(vec3)                    texture.h:18-28 */
    RT_TEX_CHECKER = 1,    /* checker_texture(even, odd)                texture.h:30-48 */
    RT_TEX_NOISE_PERLIN = 2,     /* noise_texture(PERLIN, density)      texture.h:58-59 */
    RT_TEX_NOISE_TURBULANCE = 3, /* noise_texture(TURBULANCE, density)  texture.h:60-64 */
    RT_TEX_NOISE_MARBLE = 4,     /* noise_texture(MARBLE, density)      texture.h:65-76 */
    RT_TEX_WOOD = 5,       /* wood_texture(c1, c2, density, hardness)   texture.h:86-111 */
    RT_TEX_IMAGE = 6       /* image_texture(float* rgb, w, h)           texture.h:113-148 */
};

/* acceleration structure request (the façade's bvh_node(...) is a request) */
enum {
    RT_BVH_AUTO = 0,     /* brute force for tiny scenes, host SAH for small, GPU LBVH for large */
    RT_BVH_NONE = 1,     /* hitable_list with bvh==nullptr: linear closest-hit loop (hitable_list.h:66-78) */
    RT_BVH_HOST_SAH = 2,
    RT_BVH_GPU_LBVH = 3
};

/* integrator pipeline */
enum {
    RT_PIPE_AUTO = 0,
    RT_PIPE_WAVEFRONT = 1, /* raygen / extend / per-material shade queues */
    RT_PIPE_MEGAKERNEL = 2 /* one thread runs a whole path (reference structure, main.cu:35-74) */
};

/* rt_render_params.flags.  Everything here changes the ESTIMATOR (not its expectation), so it is off by default
 * and off in every parity run against the reference (SURVEY.md 8f-4). */
#define RT_RENDER_EMITTER_SAMPLING 1u /* importance-sample the emitters at lambertian hits (the reference README's roadmap
                                        * item "Improve Sampling on emitter objects", README.md:27-28): the scatter
                                        * direction is drawn from a 50/50 mixture of the reference's n + unit-ball
                                        * distribution (material.h:112) and uniform cones towards the emitter spheres;
                                        * the path value is weighted by p_reference / p_mixture (<= 2), so the image
                                        * converges to the frame rendered without the flag */
#define RT_MAX_LIGHTS 16u             /* emitter spheres that are importance-sampled (first ones in list order) */
#define RT_MAX_CHECKER_DEPTH 8        /* checker levels a texture may nest (checker of a checker ...) above its leaf; the
                                       * shading code resolves at most this many, and rt_scene_create refuses deeper
                                       * chains (RT_ERR_UNSUPPORTED) and cycles (RT_ERR_INVALID_ARG) */

#define RT_SPHERE_MOVING 1u /* built by moving_sphere(...) (sphere.h:30-58) */
#define RT_SPHERE_INSIDE 2u /* sphere(..., inside=true); stored, no effect (sphere.h:27,133-138) */

/* sphere(center, radius, material) / moving_sphere(c0, c1, t0, t1, radius, material) */
typedef struct rt_sphere {
    float center0[3];
    float radius;
    float center1[3]; /* == center0 for a static sphere */
    float time0;
    float time1;
    uint32_t material; /* index into rt_scene_desc.materials */
    uint32_t id;       /* the reference's set_id() value (hitable_object.h:78-79) */
    uint32_t flags;    /* RT_SPHERE_* */
} rt_sphere;

typedef struct rt_material {
    uint32_t kind;   /* RT_MAT_* */
    int32_t texture; /* lambertian albedo / emitter texture; -1 otherwise */
    float albedo[3]; /* metal albedo / dielectric tint */
    float param;     /* metal: roughness (clamped to <=1 at construction); dielectric: ri; emitter: intensity */
} rt_material;

/* A checker's children may be checkers themselves (texture.h:41-48 recurses).  rt_scene_create checks every texture of
 * the description, used or not: a chain of more than RT_MAX_CHECKER_DEPTH checker levels is RT_ERR_UNSUPPORTED (the
 * reference renders it; this library declines it rather than render it wrong), a checker that reaches itself is
 * RT_ERR_INVALID_ARG (the reference cannot render it).  Both messages name the texture. */
typedef struct rt_texture {
    uint32_t kind;   /* RT_TEX_* */
    int32_t even;    /* checker: texture index used when sines >= 0 */
    int32_t odd;     /* checker: texture index used when sines <  0 */
    int32_t image;   /* image: index into rt_scene_desc.images */
    float color1[3]; /* constant: colour; wood: color1 */
    float color2[3]; /* wood: color2 */
    float density;   /* noise / wood (<=0 is replaced by 4 at construction) */
    float hardness;  /* wood */
} rt_texture;

/* image_texture(float* buffer, int width, int height): row 0 = top, RGB floats */
typedef struct rt_image {
    const float* rgb; /* width*height*3 floats, borrowed until rt_scene_create returns */
    int32_t width;
    int32_t height;
} rt_image;

/* camera(lookfrom, lookat, up, vfov, aspect, aperture, focus_dist, time0, time1), camera.h:7-10 */
typedef struct rt_camera {
    float lookfrom[3];
    float lookat[3];
    float up[3];
    float vfov; /* degrees, top to bottom */
    float aspect;
    float aperture;
    float focus_dist;
    float time0;
    float time1;
} rt_camera;

typedef struct rt_scene_desc {
    const rt_sphere* spheres;
    uint32_t n_spheres;
    const rt_material* materials;
    uint32_t n_materials;
    const rt_texture* textures;
    uint32_t n_textures;
    const rt_image* images;
    uint32_t n_images;
    rt_camera camera;
    uint32_t bvh_mode; /* RT_BVH_* */
} rt_scene_desc;

/* ---- render parameters -------------------------------------------------- */

/* The reference bakes these in: WIDTH/HEIGHT/RAY_BOUNCES/SEED (common.h:13-20),
 * SAMPLES_PER_PIXEL (main.cu:15), tmin 1e-5f (main.cu:45), world colour
 * (1,.8,.7) (main.cu:40) and the +0.1 "bloom" (main.cu:49). */
typedef struct rt_render_params {
    int32_t width;
    int32_t height;
    int32_t spp;           /* samples rendered by THIS call */
    int32_t sample_offset; /* first global sample index (multi-GPU sample sharding) */
    int32_t max_depth;     /* RAY_BOUNCES, 50 */
    uint32_t seed;         /* SEED, 1000 */
    float tmin;            /* 1e-5f */
    float world[3];        /* (1, .8, .7) */
    float bloom;           /* 0.1f */
    uint32_t pipeline;     /* RT_PIPE_* */
    uint32_t flags;        /* RT_RENDER_*, 0 = the reference's estimator */
} rt_render_params;

typedef struct rt_stats {
    uint64_t paths;    /* width*height*spp */
    uint64_t rays;     /* scene.hit() queries: primary + scattered */
    float ms_total;    /* device time, first raygen .. last accumulate (CUDA events) */
    float ms_tonemap;  /* device time of the tonemap pass (0 if not run) */
    float ms_h2d;      /* not used by render; scene upload reports it via rt_scene_info */
    float ms_d2h;      /* device->host copy of the result, if any */
    uint32_t launches; /* kernels launched by this call */
    uint32_t iterations; /* wavefront bounce iterations (1 for the megakernel) */
} rt_stats;

typedef struct rt_scene_info {
    uint32_t n_spheres;
    uint32_t n_nodes;    /* BVH nodes (0 for brute force) */
    uint32_t bvh_mode;   /* resolved RT_BVH_* */
    uint32_t bvh_depth;
    float ms_build;      /* host SAH build (wall) or device LBVH build (events) */
    float ms_upload;     /* H2D copies + device-side scene preparation */
    float sah_cost;
    uint64_t device_bytes;
} rt_scene_info;

/* ray / hit records of the parity hook */
typedef struct rt_ray {
    float origin[3];
    float direction[3]; /* NOT normalised (ray.h:12, camera.h:37) */
    float time;
} rt_ray;

typedef struct rt_hit {
    float t;      /* FLT_MAX on miss */
    uint32_t id;  /* rt_sphere.id of the closest object, RT_INVALID_ID on miss */
    float p[3];
    float n[3];   /* outward normal (sphere.h:123) */
    float u, v;   /* get_sphere_uv (sphere.h:61-83), computed for every sphere kind.
                   * DELIBERATE DEVIATION from the reference: moving_sphere::hit (sphere.h:157-190) never writes
                   * u and v, so the reference shades a moving sphere with whatever the shared temp_rec of its
                   * traversal loop last held (hitable_list.h:69-76, bvh.h:130-150) — the (u, v) of the last
                   * static sphere whose hit() succeeded on that ray in ITS traversal order, or uninitialised
                   * stack memory when there was none.  That value depends on the reference's BVH topology
                   * (random split axes, bvh.h:84-92) and, in the second case, on nothing at all, so it cannot be
                   * reproduced by another acceleration structure; this library computes the moving sphere's own
                   * (u, v) at the ray's time.  Only an IMAGE texture on a MOVING sphere can tell the difference
                   * (none of the reference's scenes has one); the oracle (oracle/rt_oracle.cpp) restates the
                   * reference's list-order behaviour and the parity tests mask moving spheres out of the (u, v)
                   * comparison (tests/test_gpu_parity.py). */
} rt_hit;

/* One integrator step at the closest hit of a caller-supplied ray (second parity hook): the terms of
 * color()'s loop body, main.cu:45-55.  The step draws its random numbers with the Philox key
 * (pixel = ray index, sample = 0, bounce = 1). */
typedef struct rt_shade_sample {
    uint32_t id;          /* closest object, RT_INVALID_ID on miss (everything below is then 0) */
    uint32_t continues;   /* 1: material::scatter returned true and `scattered` is valid; 0: the path ends with `emitted` */
    float t;
    float emitted[3];     /* m.emit(h) + bloom (main.cu:49) */
    float attenuation[3]; /* scatter()'s attenuation (main.cu:50-51) */
    rt_ray scattered;     /* origin = hit point, direction NOT normalised, time (material.h:113,125,179-181) */
} rt_shade_sample;

typedef struct rt_context rt_context;
typedef struct rt_scene rt_scene;

/* ---- entry points -------------------------------------------------------- */

int rt_api_version(void);
/* sizeof() of a structure of this header by name ("rt_sphere", ...), 0 if unknown: lets a
 * foreign-language binding verify its layout before passing memory across the boundary. */
size_t rt_abi_sizeof(const char* struct_name);
const char* rt_last_error(void);
void rt_default_render_params(rt_render_params* p); /* reference constants, 1200x600x100 */

/* One context = one CUDA device + one stream (one process per GPU). Replaces
 * the implicit device-0/default-stream use of main() (main.cu:368-509). */
rt_status rt_context_create(int device, rt_context** out);
void rt_context_destroy(rt_context* ctx);
/* run on a caller-owned stream (e.g. torch's current stream) instead of the context's own */
rt_status rt_context_set_stream(rt_context* ctx, void* cuda_stream);
rt_status rt_context_synchronize(rt_context* ctx);

/* Replaces populate_scene_balls<<<1,1>>> (main.cu:188-356, :423) + the image
 * upload (main.cu:383-388): copies the POD scene to the device, prepares the
 * SoA sphere arrays and builds the acceleration structure. */
rt_status rt_scene_create(rt_context* ctx, const rt_scene_desc* desc, rt_scene** out);
/* A scene belongs to its context (device memory comes from the context's stream-ordered pool and is
 * released on the context stream): destroy scenes before their context.  A scene may be RENDERED through another
 * context of the same device (frame pipelines: one context uploads scene k+1 on its stream while another renders
 * frame k); the caller then destroys a scene only after the frames that use it have completed.  Contexts may be used
 * from different host threads at the same time; one context is used by one thread at a time. */
void rt_scene_destroy(rt_scene* scene); /* replaces free_scene<<<1,1>>> (main.cu:360-366) */
rt_status rt_scene_get_info(const rt_scene* scene, rt_scene_info* info);

/* An edit of a resident scene.  Indices are positions in the rt_scene_desc the scene was created from. */
typedef struct rt_scene_edit {
    const uint32_t* sphere_index;   /* spheres to replace (list ordinals), each at most once per edit */
    const rt_sphere* spheres;       /* their new values */
    uint32_t n_spheres;
    const uint32_t* material_index; /* materials to replace, each at most once per edit */
    const rt_material* materials;   /* their new values */
    uint32_t n_materials;
    const rt_camera* camera;        /* NULL: keep the scene's camera */
} rt_scene_edit;
/* Applies an edit to a scene on the device, without a new upload or build.  After RT_OK the scene renders and probes
 * exactly like rt_scene_create of its creation description with the edit applied (same bvh_mode): rt_trace_primary gives
 * bit-identical hits for every use_bvh both scenes support, rt_shade_probe identical records, renders equal sample and
 * ray counts and sums equal up to the order of float additions.  The tree keeps its topology and depth; every node box is
 * refitted on the device (all node forms), so large motions make the tree slower, never wrong — create the scene again
 * for a fresh tree.  rt_scene_get_info keeps describing the scene as it was built.
 * Not editable: the sphere and material counts, textures, images, bvh_mode, and a sphere's RT_SPHERE_MOVING flag (static
 * spheres are stored first; create a sphere that may start moving as a moving sphere with center1 == center0).
 * Every argument is checked before any device work; RT_ERR_INVALID_ARG leaves the scene unchanged: NULLs, ctx not the
 * scene's own context, indices out of range or repeated, a changed RT_SPHERE_MOVING flag, and the sphere, material and
 * camera rules of rt_scene_create.  An empty edit is a valid no-op.
 * Ordering: the update runs on ctx's stream after the work queued there before it (a render enqueued before the call
 * renders the old scene); renders of this scene through other contexts must have completed (as for rt_scene_destroy).
 * Returns when the update is complete.  ms_device (may be NULL): device time of the update.  A CUDA error during the
 * update (RT_ERR_CUDA / RT_ERR_OOM) leaves the scene unusable: destroy it. */
rt_status rt_scene_update(rt_context* ctx, rt_scene* scene, const rt_scene_edit* edit, float* ms_device);
/* rt_scene_update of an edit that has only spheres, read from DEVICE memory: for a simulation whose sphere state lives on
 * the GPU (no copy to the host and back per step).  The records are checked, packed and scattered on the device; after
 * RT_OK the scene equals rt_scene_create of its description with the edit applied, and what rt_scene_update of the same
 * records gives.  Materials and the camera stay with rt_scene_update.
 * sphere_index_dev: n_spheres list ordinals (uint32, 4-byte aligned); spheres_dev: n_spheres rt_sphere records (16-byte
 * aligned).  Both are device or managed memory of ctx's device and at least n_spheres elements long (not checkable: the
 * caller's guarantee).  n_spheres = 0 is a valid no-op without device work; the pointers may then be NULL.
 * Checked on the host before any device work: NULLs, ctx not the scene's context, a pointer that is not device or managed
 * memory of ctx's device (never handed to a kernel), the alignments.  Checked on the device before anything of the scene
 * is written: the sphere rules of rt_scene_update (index in range, not repeated, RT_SPHERE_MOVING unchanged, material in
 * range, centre / radius / times finite).  The failure reported is the one rt_scene_update would report: the lowest
 * failing position, its first rule in that order.  RT_ERR_INVALID_ARG leaves the scene unchanged.
 * Ordering: the records are read on ctx's stream after the work queued there before the call (a render enqueued before
 * the call renders the old scene).  Records written on another stream (e.g. torch's current stream) must be ordered
 * before the call by the caller: rt_context_set_stream to that stream, or a synchronise.  Returns when the update is
 * complete; the caller may then overwrite both buffers.  ms_device and CUDA errors: as for rt_scene_update. */
rt_status rt_scene_update_device(rt_context* ctx, rt_scene* scene, const uint32_t* sphere_index_dev,
                                 const rt_sphere* spheres_dev, uint32_t n_spheres, float* ms_device);

/* Parity hook: closest hit of scene.hit(r, tmin, FLT_MAX) (hitable_list.h:60-79)
 * for n caller-supplied rays.  use_bvh = 0 forces the brute-force list path, 1 walks the binary BVH
 * (bvh_node::dfs, bvh.h:121-155), 2 the 4-wide form of the same tree, 3 its 64-byte quantised form — the nodes the
 * large-scene render kernel traverses (RT_ERR_INVALID_ARG when the scene has none). */
rt_status rt_trace_primary(rt_context* ctx, const rt_scene* scene, const rt_ray* rays, size_t n,
                           float tmin, int use_bvh, rt_hit* hits);

/* Self-test of the renderer's own round-toward-zero division and square root (csrc/rt_device.cuh: the reference's vec3
 * operator/ and length() are __fdiv_rz / __fsqrt_rz, vec3.h:153-166,334-347; the library computes them from the
 * round-to-nearest forms and one exact FMA residual): out[4i .. 4i+3] = { div_rz(x, y), __fdiv_rz(x, y), sqrt_rz(x),
 * __fsqrt_rz(x) } for n caller-supplied operand pairs (HOST arrays), so a test can require bit equality. */
rt_status rt_selftest_rz(rt_context* ctx, const float* x, const float* y, size_t n, float* out);

/* Self-tests of the device-wide primitives the LBVH build, the 4-wide compaction, the adaptive pixel list and the JPEG
 * writer are built on (csrc/rt_prims.cuh), with HOST arrays in and out.  Each call allocates its device buffers and the
 * primitive's scratch from the context's pool with the sizes the library's own callers use, puts 256 bytes of 0xA5
 * before and after every buffer the primitive may write, and sets *overrun to 1 if any of those bytes changed, else 0.
 * Arguments are checked before any device work; n = 0 is valid, launches nothing and writes no output array.
 * Exclusive prefix sum of n unsigned integers of elem_bytes (4 or 8) bytes, wrapping like the integer type:
 * out[i] = in[0] + ... + in[i-1].  in_place != 0 scans one device buffer in place, else from an input buffer into an
 * output buffer. */
rt_status rt_selftest_exclusive_sum(rt_context* ctx, const void* in, void* out, size_t n, int32_t elem_bytes, int32_t in_place,
                                    int32_t* overrun);
/* Stable LSD radix sort of n (64-bit key, 32-bit value) pairs by the key bits [0, 8*passes), passes in [1, 8], n < 2^32:
 * keys_out / vals_out receive the sorted pairs with their full keys; *in_alt = 1 when the result came out of the
 * ping-pong buffers (an odd number of passes). */
rt_status rt_selftest_sort_pairs(rt_context* ctx, const uint64_t* keys, const uint32_t* vals, size_t n, int32_t passes,
                                 uint64_t* keys_out, uint32_t* vals_out, int32_t* in_alt, int32_t* overrun);

/* Second parity hook: closest hit + one shading step per ray (see rt_shade_sample). */
rt_status rt_shade_probe(rt_context* ctx, const rt_scene* scene, const rt_ray* rays, size_t n,
                         const rt_render_params* p, int use_bvh, rt_shade_sample* out);

/* Replaces init_rand_state + render (main.cu:76-132, :438-449). out_rgb is a
 * HOST buffer of width*height*3 floats in the reference framebuffer layout:
 * index j*width+i, j=0 = bottom row, values /spp, saturated, sqrt-gamma'd. */
rt_status rt_render(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                    float* out_rgb, rt_stats* stats);

/* Un-tonemapped per-pixel sums: HOST buffer of width*height*4 floats
 * (sum r, sum g, sum b, sample count). */
rt_status rt_render_accum(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                          float* out_accum, rt_stats* stats);

/* Device-resident variant: ADDS this call's samples into accum_dev (float4 per
 * pixel, caller-allocated device memory, caller zeroes it). Asynchronous on the
 * context stream unless stats != NULL (then it synchronises to fill stats). */
rt_status rt_render_accum_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                                 void* accum_dev, rt_stats* stats);

/* Progressive accumulation (SURVEY.md 8f-4; the reference's README "interactive" roadmap item, README.md:25-26):
 * `passes` passes of p->spp samples each are added to ONE accumulator; after every pass the frame is finalised
 * (the accumulator carries the per-pixel sample count) into out_rgb (HOST, layout of rt_render) and `on_pass`
 * (may be NULL) is called with the pass index and the samples per pixel so far; a non-zero return stops early.
 * Pass k uses sample indices [offset + k*spp, offset + (k+1)*spp): the final frame is the frame rt_render
 * produces with passes*spp samples, up to the order of float additions. */
typedef int (*rt_progress_fn)(int32_t pass, int32_t spp_so_far, const float* rgb, void* user);
rt_status rt_render_progressive(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t passes,
                                float* out_rgb, rt_progress_fn on_pass, void* user, rt_stats* stats);

/* Pixel finalisation of main.cu:124-127 on the device: col * rz(1/count) ->
 * saturate -> sqrt. out_rgb_dev: width*height*3 floats (reference layout) or NULL;
 * out_rgb8_dev: width*height*3 bytes, Y-flipped and quantised as main.cu:476-487, or NULL. */
rt_status rt_tonemap_device(rt_context* ctx, const void* accum_dev, int32_t width, int32_t height,
                            void* out_rgb_dev, void* out_rgb8_dev);

/* Multi-GPU finalisation fused with the collective, over NVLink peer memory (one process per GPU, the
 * accumulators allocated as symmetric memory so every rank holds device pointers to every rank's copy):
 * for rows [row_begin, row_end) sums the n_peers accumulators — with NVLS `multimem.ld_reduce` on
 * `multicast_accum` when it is not NULL, else with peer loads added in rank order — and applies the pixel
 * finalisation of rt_tonemap_device to the sum.  Outputs may be peer pointers (e.g. the root's image);
 * out_sum_dev (may be NULL) receives the summed float4 accumulator.  The caller orders this kernel after
 * every rank's render (a symmetric-memory barrier) and before the root reads the image (a second one). */
rt_status rt_reduce_tonemap_peers(rt_context* ctx, const void* const* peer_accum_dev, int32_t n_peers,
                                  const void* multicast_accum, int32_t width, int32_t height, int32_t row_begin,
                                  int32_t row_end, void* out_rgb_dev, void* out_rgb8_dev, void* out_sum_dev);

/* ---- denoiser -------------------------------------------------------------------------------------------------
 * A post-pass over the float4 accumulator of any render entry: first-hit feature buffers and the edge-avoiding à-trous
 * wavelet filter (Dammertz et al., HPG 2010), then the pixel finalisation of rt_tonemap_device.  No render kernel is
 * involved.
 * Features: 2*width*height float4, two planes in the accumulator's layout (index j*width+i, j = 0 the bottom row):
 *   plane 0 [0, W*H):      mean outward unit normal (not renormalised) and mean hit distance t*|d| over the camera
 *                          samples that hit (0 when none does);
 *   plane 1 [W*H, 2*W*H):  mean albedo over all samples (scatter()'s attenuation; emit for an emitter; the world colour
 *                          for a miss) and the fraction of samples that hit.
 * Filter level i (0 <= i < iterations) is a 5x5 B3-spline kernel with taps 2^i pixels apart, each tap weighted by
 *   exp(-|c_p-c_q|^2/(sigma_color 2^-i)^2) exp(-|n_p-n_q|^2/sigma_normal^2) exp(-|z_p-z_q|/(sigma_depth max(z_p,z_q,1e-4)))
 *   exp(-(|a_p-a_q|^2 + (f_p-f_q)^2)/sigma_albedo^2)
 * on the mean colour accum.rgb/accum.w saturated to [0, 1].  Pixels without samples are finalised as rt_tonemap_device
 * finalises them.  The colour is not divided by the albedo: the estimator's first-hit attenuation multiplies only what the
 * path gathers after that hit, not the pixel value. */
typedef struct rt_denoise_params {
    int32_t iterations;  /* à-trous levels, 0..8; 0 = no filtering (== rt_tonemap_device) */
    int32_t feature_spp; /* camera samples per pixel of the feature pass, >= 1 */
    float sigma_color, sigma_normal, sigma_depth, sigma_albedo; /* > 0, finite */
} rt_denoise_params;
void rt_default_denoise_params(rt_denoise_params* d); /* 3 levels, 4 feature samples, sigmas 0.5, 1, 0.3, 1 */
/* features of p's camera samples [p->sample_offset, p->sample_offset + feature_spp) into features_dev (device memory,
 * layout above); p->spp is not used.  Asynchronous on the context stream. */
rt_status rt_render_features_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                                    int32_t feature_spp, void* features_dev);
/* filter + finalisation of a device accumulator: out_rgb_dev / out_rgb8_dev (either may be NULL, not both) as
 * rt_tonemap_device writes them.  Asynchronous on the context stream; scratch comes from the context's memory pool. */
rt_status rt_denoise_device(rt_context* ctx, const void* accum_dev, const void* features_dev, int32_t width,
                            int32_t height, const rt_denoise_params* d, void* out_rgb_dev, void* out_rgb8_dev);
/* rt_render + features (d->feature_spp samples from p->sample_offset) + filter + finalisation; out_rgb: HOST, layout of
 * rt_render.  stats->ms_tonemap = device time of features + filter + finalisation. */
rt_status rt_render_denoised(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                             const rt_denoise_params* d, float* out_rgb, rt_stats* stats);

/* ---- adaptive sampling --------------------------------------------------------------------------------------------
 * Pixels stop sampling once their noise estimate falls below a threshold.  Pass 0 gives every pixel min_spp samples; each
 * later pass gives step_spp samples to the pixels still listed, until the list is empty or max_spp is reached.  A path
 * adds into plane A (even samples, counted from p->sample_offset) or plane B (odd samples) of a two-plane accumulator
 * (2*W*H float4: plane A, then plane B).  After every pass but the last, the error of pixel p is, with g(x) =
 * sqrt(saturate(x)),
 *   e_p = (|g(A_r/A_w) - g(B_r/B_w)| + |g(A_g/A_w) - g(B_g/B_w)| + |g(A_b/A_w) - g(B_b/B_w)|) / 6      (+inf if A_w or B_w = 0)
 * (half the mean over the channels of the difference of the two half means: the standard error of the full mean in
 * display space), the windowed error ebar_p = (sum of e over the 3x3 neighbourhood, coordinates clamped to the frame,
 * in row-major order) / 9, every step one IEEE float operation, and the list keeps, in its order (pixel order), the pixels
 * with ebar_p >= threshold and count(p) < max_spp.  A pixel that stopped never restarts, so pixel p has exactly the samples
 * [p->sample_offset, p->sample_offset + count(p)), count(p) = min_spp + k*step_spp: the samples a uniform render of
 * count(p) spp gives it.  Stopping early carries the small bias of every adaptive sampler; threshold = 0 removes it. */
typedef struct rt_adaptive_params {
    int32_t min_spp;  /* first pass, every pixel; even, >= 2 */
    int32_t step_spp; /* every later pass, listed pixels only; even, >= 2 */
    int32_t max_spp;  /* cap: min_spp + k*step_spp for some k >= 0, <= 2^24 */
    float threshold;  /* display-space standard-error target, finite, >= 0; 0 = never stop early */
} rt_adaptive_params;
void rt_default_adaptive_params(rt_adaptive_params* a); /* min 32, step 32, max 256, threshold 1/255 */
/* windowed error map (ebar above) of a two-plane accumulator (2*W*H float4, device) into error_dev (W*H floats, device).
 * Asynchronous on the context stream. */
rt_status rt_adaptive_error_device(rt_context* ctx, const void* planes_dev, int32_t width, int32_t height, void* error_dev);
/* p->spp is not used; samples start at p->sample_offset.  accum_dev (W*H float4, device) is WRITTEN (A + B), not added to;
 * error_dev (W*H floats, device, may be NULL) receives the final windowed error; *passes (may be NULL) the passes run.
 * stats (may be NULL): paths = samples actually traced, rays, launches, iterations, ms_total = device time of the whole
 * call.  Returns when the frame is finished (the planes and lists live in the context's memory pool). */
rt_status rt_render_adaptive_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                                    const rt_adaptive_params* a, void* accum_dev, void* error_dev, int32_t* passes,
                                    rt_stats* stats);
/* host convenience: out_rgb (HOST) as rt_render writes it; out_spp (HOST, may be NULL) W*H int32 samples per pixel in the
 * same layout */
rt_status rt_render_adaptive(rt_context* ctx, const rt_scene* scene, const rt_render_params* p,
                             const rt_adaptive_params* a, float* out_rgb, int32_t* out_spp, rt_stats* stats);

/* ---- frame sequences ----------------------------------------------------------------------------------------------
 * n_frames frames of one scene in one render: frame f looks through cameras[f] (its time0 / time1 shutter included; the
 * scene's own camera is not used) and takes the sample indices [p->sample_offset + f*p->spp, p->sample_offset +
 * (f+1)*p->spp), the convention of rt_render_progressive's passes: frames have independent noise under the same seed.
 * So frame f is the frame rt_render_accum_device gives on a scene whose camera is cameras[f] with sample_offset =
 * p->sample_offset + f*p->spp: equal sample counts and ray counts, sums equal up to the order of float additions.  Every
 * pipeline and RT_RENDER_EMITTER_SAMPLING work as for one frame.  The paths of all frames share one wavefront, so the
 * next frame's paths fill the thin end of the previous one.  The scene is not re-uploaded; the cameras are (n_frames *
 * 84 bytes).  Checked before any device work: NULLs, n_frames >= 1, p, every camera finite, and sample_offset +
 * n_frames*spp <= 2^31 - 1. */
/* ADDS frame f's samples into accum_dev + f*W*H (n_frames*W*H float4, device, caller zeroes it).  Asynchronous on the
 * context stream unless stats != NULL; stats: paths = W*H*spp*n_frames, rays, launches, iterations and ms_total of the
 * whole batch. */
rt_status rt_render_frames_device(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_camera* cameras,
                                  int32_t n_frames, void* accum_dev, rt_stats* stats);
/* host convenience: out_rgb (HOST) n_frames*W*H*3 floats, frame f from f*W*H*3 on in rt_render's layout; ms_tonemap is the
 * finalisation of all frames */
rt_status rt_render_frames(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, const rt_camera* cameras,
                           int32_t n_frames, float* out_rgb, rt_stats* stats);
/* Cameras of an orbit or a motion sequence (no device needed).  Frame k (0 <= k < n_frames) is *base with lookfrom rotated by
 * k*degrees/n_frames degrees about the axis through lookat along up (right-hand rule) and the shutter
 * [t0 + k*(t1-t0)/n_frames, t0 + (k+1)*(t1-t0)/n_frames] of base's [t0, t1] = [time0, time1]: the frames' windows tile
 * base's.  Computed in double and rounded to float once.  degrees = 0 keeps lookfrom: the frames of a still camera over
 * successive shutter windows.  Checks: NULLs, n_frames >= 1, degrees and base finite, up not zero. */
rt_status rt_orbit_cameras(const rt_camera* base, int32_t n_frames, float degrees, rt_camera* out);

/* ---- multi-GPU (SURVEY.md 8e; BASELINE.json north_star (4))---------------------------------------------------
 * Samples per pixel are split across the GPUs of one box: GPU r renders sample indices [first_r, first_r + count_r) of
 * EVERY pixel (rt_render_params.sample_offset; the Philox keys use the global sample index, so the image does not depend
 * on the number of GPUs) into its own float4 accumulator; the accumulators are summed in rank order and finalised by
 * one fused kernel per GPU that reads the peers' accumulators over NVLink and writes its band of rows into the root's
 * image.  The reference's main() (main.cu:368-509) is a single-device program: these entries are what its device
 * selection, cudaMallocManaged frame buffer and render launch become on an 8-GPU box. */
/* contiguous sample ranges, the remainder spread over the low ranks; row bands of the fused reduce (no device needed) */
rt_status rt_shard_samples(int32_t spp_total, int32_t rank, int32_t world, int32_t* first, int32_t* count);
rt_status rt_shard_rows(int32_t height, int32_t rank, int32_t world, int32_t* row_begin, int32_t* row_end);

/* (a) ONE process, n devices.  devices == NULL / n_devices <= 0: every visible device.  Creates a context per device
 * and enables peer access between all of them (RT_ERR_UNSUPPORTED without a P2P path). */
typedef struct rt_multi rt_multi;
rt_status rt_multi_create(const int32_t* devices, int32_t n_devices, rt_multi** out);
int32_t rt_multi_size(const rt_multi* m);
/* uploads the scene to every device (the uploads and BVH builds run side by side) */
rt_status rt_multi_set_scene(rt_multi* m, const rt_scene_desc* desc);
/* rt_scene_update of every member's scene with the same edit (the updates run side by side); reports the first failing
 * device */
rt_status rt_multi_update_scene(rt_multi* m, const rt_scene_edit* edit);
/* p->spp is the TOTAL sample count of the frame.  out_rgb (HOST, layout of rt_render) and/or out_rgb8 (HOST, Y-flipped
 * bytes as main.cu:476-487).  stats (may be NULL): paths, rays and launches summed over the devices, ms_total = the slowest
 * device's render, ms_tonemap = device time from the root's render end to the last band of the reduce, ms_d2h = wall
 * clock of the whole call.  ms_reduce (may be NULL) = stats->ms_tonemap. */
rt_status rt_multi_render(rt_multi* m, const rt_render_params* p, float* out_rgb, uint8_t* out_rgb8, rt_stats* stats, float* ms_reduce);
/* the un-finalised float4 accumulator of one member after rt_multi_render (HOST, the size of the largest frame rendered
 * so far): lets a caller check the fused reduce against its own rank-ordered sum */
rt_status rt_multi_read_accum(rt_multi* m, int32_t member, float* out_accum);
void rt_multi_destroy(rt_multi* m);

/* (b) one PROCESS per GPU (torchrun, MPI, ...): `world` members, member `rank` lives on ctx's device.  Every member
 * allocates its accumulator (and member 0 the image) with cudaMalloc and exports it as a CUDA IPC handle; the caller
 * gathers the RT_GROUP_HANDLE_BYTES blobs of all members in rank order by any means it has and passes the table to
 * rt_group_connect.  Per frame, on every member:
 *     rt_group_begin_frame(g);                                   zero the accumulator
 *     rt_render_accum_device(ctx, scene, &p_shard, rt_group_accum(g), NULL);      p_shard from rt_shard_samples
 *     rt_group_finish_frame(g, want_rgb8, NULL);                 barrier, fused reduce + finalisation of this member's band, barrier
 *     rt_group_read_frame(g, out_rgb, out_rgb8);                 member 0: D2H of the image; every member: synchronise
 * All of it is stream-ordered on the context's stream; the two barriers are flag exchanges in peer memory (every member
 * runs on its own GPU).  A member that never arrives turns into RT_ERR_CUDA from rt_group_read_frame after a few
 * seconds instead of a hung GPU.  ms_reduce (may be NULL; synchronises): device time of barrier + reduce + barrier. */
typedef struct rt_group rt_group;
#define RT_GROUP_HANDLE_BYTES 192
rt_status rt_group_create(rt_context* ctx, int32_t rank, int32_t world, int32_t width, int32_t height, rt_group** out);
rt_status rt_group_export(const rt_group* g, void* handle);
rt_status rt_group_connect(rt_group* g, const void* handles);
void* rt_group_accum(const rt_group* g);
rt_status rt_group_begin_frame(rt_group* g);
rt_status rt_group_finish_frame(rt_group* g, int32_t want_rgb8, float* ms_reduce);
rt_status rt_group_read_frame(rt_group* g, float* out_rgb, uint8_t* out_rgb8);
rt_status rt_group_read_accum(rt_group* g, float* out_accum); /* this member's float4 accumulator (HOST, width*height*4 floats) */
void rt_group_destroy(rt_group* g);

/* Host restatement of the writer loop main.cu:475-488 (Y flip + int(255.999f*c)&255). */
rt_status rt_quantize_rgb8(const float* rgb, int32_t width, int32_t height, uint8_t* out_rgb8);
rt_status rt_write_ppm(const char* path, int32_t width, int32_t height, const uint8_t* rgb8);
rt_status rt_read_ppm_f32(const char* path, float** out_rgb, int32_t* width, int32_t* height); /* P6 or P5, byte/255.f */
/* Image-texture ingest (SURVEY.md 8f-2): the `channels`-component float image stbi_loadf returns (main.cu:376-380;
 * the reference assumes 3, texture.h:118-132) as the RGB image rt_image carries: grey / grey+alpha replicate the
 * grey value, RGBA drops alpha.  Any width x height is accepted by rt_scene_create (the reference passes the RENDER
 * size as the texture size, main.cu:237). */
rt_status rt_image_to_rgb(const float* data, int32_t width, int32_t height, int32_t channels, float* out_rgb);
void rt_free(void* p);

/* ---- output stage (SURVEY.md 8f-1) ------------------------------------------------------------------
 * Replaces stbi_write_jpg("render.jpg", W, H, 3, data, 100) (main.cu:491; vendored stb_image_write v1.15,
 * stb_image_write.h:1368-1573) with CUDA kernels whose output is byte-identical to stb's for the same
 * pixels and quality (1..100; <= 90 selects 4:2:0 chroma subsampling exactly like stb).
 * `rgb8` is what the reference hands to stb: height rows of width RGB bytes, first row = top of the picture
 * (rt_tonemap_device's out_rgb8_dev / rt_quantize_rgb8). */
size_t rt_jpeg_max_bytes(int32_t width, int32_t height); /* capacity that always suffices */
/* device image -> finished file in HOST memory; out_jpg == NULL only reports *n_bytes.  ms_device (may be NULL)
 * receives the device time of the encoder passes. */
rt_status rt_jpeg_encode_device(rt_context* ctx, const void* rgb8_dev, int32_t width, int32_t height, int32_t quality,
                                uint8_t* out_jpg, size_t cap, size_t* n_bytes, float* ms_device);
/* host image -> H2D -> encode -> D2H */
rt_status rt_jpeg_encode(rt_context* ctx, const uint8_t* rgb8, int32_t width, int32_t height, int32_t quality,
                         uint8_t* out_jpg, size_t cap, size_t* n_bytes);
/* stbi_write_jpg(filename, w, h, 3, data, quality) */
rt_status rt_write_jpg(rt_context* ctx, const char* path, int32_t width, int32_t height, const uint8_t* rgb8, int32_t quality);
/* render + pixel finalisation + Y flip + quantisation + JPEG, all on the device: only the file crosses PCIe
 * (main.cu:442-491 in one call).  stats->ms_d2h reports the device time of the JPEG passes. */
rt_status rt_render_jpeg(rt_context* ctx, const rt_scene* scene, const rt_render_params* p, int32_t quality,
                         uint8_t* out_jpg, size_t cap, size_t* n_bytes, rt_stats* stats);

/* ---- JPEG reader (SURVEY.md 8f-2) --------------------------------------------------------------------
 * Replaces stbi_loadf(path, &w, &h, &ch, 0) with ldr_to_hdr gamma = scale = 1 (main.cu:376-380; vendored stb_image
 * v2.26) for baseline and progressive 8-bit JPEG files with 1 or 3 components: the Huffman decoding stays on the
 * host (a serial bit stream), dequantisation + IDCT + chroma up-sampling + YCbCr->RGB + byte/255.f run on the GPU.
 * The float image equals stb's bit for bit. */
typedef struct rt_jpeg_component {
    int32_t h, v, tq;             /* sampling factors, quantiser index */
    int32_t x, y;                 /* effective pixels of the component */
    int32_t w2, h2;               /* plane size padded to whole MCUs */
    int32_t blocks_w, blocks_h;   /* w2 / 8, h2 / 8 */
    const int16_t* coeff;         /* blocks_w * blocks_h * 64 coefficients, row-major inside a block, not dequantised */
} rt_jpeg_component;
typedef struct rt_jpeg_coefficients {
    int32_t width, height, n_comp, h_max, v_max, progressive, is_rgb;
    rt_jpeg_component comp[3];
    uint16_t dequant[4][64];      /* row-major order */
} rt_jpeg_coefficients;
/* host half only (no device needed): the decoded coefficient planes; release with rt_jpeg_coefficients_free */
rt_status rt_jpeg_parse(const uint8_t* file, size_t n_bytes, rt_jpeg_coefficients** out);
void rt_jpeg_coefficients_free(rt_jpeg_coefficients* c);
/* whole reader: *out_pixels = malloc'd width*height*channels floats (channels 3, or 1 for a grey file), first row =
 * top of the picture; release with rt_free.  ms_device (may be NULL): device time of the pixel stages. */
rt_status rt_jpeg_decode(rt_context* ctx, const uint8_t* file, size_t n_bytes, float** out_pixels, int32_t* width,
                         int32_t* height, int32_t* channels, float* ms_device);
/* file -> RGB floats for rt_image: JPEG through rt_jpeg_decode (+ rt_image_to_rgb for grey files), P5/P6 through
 * rt_read_ppm_f32 */
rt_status rt_image_load(rt_context* ctx, const char* path, float** out_rgb, int32_t* width, int32_t* height);

/* Built-in scene generators written against the façade (BASELINE configs C1..C4):
 * "earth_emitter" (main.cu:188-356), "hdr_sphere" (main.cu:136-182, needs an environment image), "book1_final",
 * "perlin_motion", "random_spheres".
 * `image_rgb` (may be NULL unless the scene needs it) is the earth texture; `n` is
 * the primitive count for "random_spheres" (ignored otherwise). The returned desc owns
 * its arrays; release with rt_scene_desc_free. */
rt_status rt_builtin_scene(const char* name, const float* image_rgb, int32_t image_w, int32_t image_h,
                           uint32_t n, uint32_t bvh_mode, rt_scene_desc** out);
void rt_scene_desc_free(rt_scene_desc* desc);
/* Runtime scene front-end (SURVEY.md 8f-3; replaces the compile-time scene of populate_scene_balls, main.cu:188-356,
 * and the WIDTH/HEIGHT/SAMPLES_PER_PIXEL/SEED macros, common.h:13-20, main.cu:15): a JSON document (format:
 * include/rt/scene_json.hpp) -> the same façade objects a C++ caller creates -> flattened description.
 * `base_dir` resolves relative image files (P5/P6, or JPEG through rt_image_load when `ctx` is not NULL: the pixel
 * stages of the JPEG reader run on the device); `render` (may be NULL) is updated from the "render" block.  Errors: RT_ERR_INVALID_ARG with the parser's message in rt_last_error().  Release with rt_scene_desc_free. */
rt_status rt_scene_desc_from_json(rt_context* ctx, const char* json_text, const char* base_dir, rt_render_params* render,
                                  rt_scene_desc** out);
rt_status rt_scene_desc_from_json_file(rt_context* ctx, const char* path, rt_render_params* render, rt_scene_desc** out);
/* flat binary scene file shared with the reference harness (oracle/ref_harness.cu) */
rt_status rt_scene_desc_save(const rt_scene_desc* desc, const char* path);
rt_status rt_scene_desc_load(const char* path, rt_scene_desc** out);

#ifdef __cplusplus
}
#endif
#endif /* RT_API_H */
