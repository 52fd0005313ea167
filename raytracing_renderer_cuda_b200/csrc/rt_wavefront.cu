// rt_wavefront.cu — the wavefront pipeline (BASELINE.json north_star (2)).
//
// A pool of P path slots lives in device memory as 64-byte records; every iteration ONE
// kernel launch advances every live path by one bounce.  Work is organised as queues of
// slot indices, one queue per shading class:
//
//   Q_NEW         free slots: ray-gen (camera + jitter + Philox) for the next path id
//   Q_LAMB_CONST  lambertian, constant albedo
//   Q_LAMB_NOISE1 lambertian, one-octave Perlin (noise PERLIN, wood)
//   Q_LAMB_NOISE6 lambertian, six-octave turbulence (noise TURBULANCE / MARBLE)
//   Q_LAMB_IMAGE  lambertian, image texture
//   Q_METAL, Q_DIEL
//   Q_EMIT        emitter with a non-constant texture (constant emitters and misses
//                 terminate inside the extend step: "shadow/emission")
//
// Work is handed out in chunks of consecutive entries of ONE queue, so every warp runs one shader with all
// lanes doing the same thing (the reference's megakernel mixes all of them in every warp).  The shade step
// produces the scattered ray, the same thread extends it (closest hit), classifies the hit and pushes its slot
// into the matching queue of the next iteration.  Pushes are compacted with warp ballots and aggregated into
// one global atomic per (chunk, queue); two chunk granularities exist (CTA chunks / ticketed warp chunks, see
// the two kernels below).  Terminated paths add their value to the float4 accumulator with a single vector
// reduction (RED.ADD.F32x4) and hand their slot to Q_NEW, so the pool stays full until the frame's paths run
// out (path regeneration).
//
// Pool size: measured, bigger is better up to 16 Mi slots (rt_api.cu) — the records stream through HBM at ~25 %
// of its bandwidth (ncu: 119 B per slot and iteration, the algorithmic 120 B/ray), far from being the limit.
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "rt_kernels.cuh"
#include "rt_shade.cuh"

namespace rtd {

enum : int { Q_NEW = 0, Q_LAMB_CONST, Q_LAMB_NOISE1, Q_LAMB_NOISE6, Q_LAMB_IMAGE, Q_METAL, Q_DIEL, Q_EMIT, NQ };
#define Q_NONE (-1)
#ifndef WF_THREADS
#define WF_THREADS 256
#endif
// Programmatic dependent launch: iteration i+1 is launched while iteration i drains, so its CTAs are resident and
// waiting (griddepcontrol.wait returns once the previous grid has completed and its writes are visible) instead
// of paying the launch latency between two of the ~70 dependent launches of a frame.
#define WF_PDL_PROLOGUE()                                      \
    asm volatile("griddepcontrol.launch_dependents;");          \
    asm volatile("griddepcontrol.wait;" ::: "memory")
#ifndef WF_CTA_THREADS
// CTA size of the CTA-chunk kernel (= its chunk size).  128 threads x 8 CTAs per SM instead of 256 x 4: the two block
// barriers of a chunk span 4 warps instead of 8 (C1 -1.1 % at equal table size (round-1 A/B, log not kept); 64 x 16: +2 %)
#define WF_CTA_THREADS 128
#endif
#ifndef WF_CTA_MINBLOCKS
#define WF_CTA_MINBLOCKS (WF_THREADS * 4 / WF_CTA_THREADS) // 64 registers/thread: 32 warps per SM
#endif
#ifndef WF_MINBLOCKS
#define WF_MINBLOCKS 4 // 64 registers/thread: 32 warps per SM (A/B on C1: 15.4 ms at 2, 13.5 at 3, 12.6 at 4)
#endif

struct WfRecord { // 64 B, one per slot
    float4 o;     // origin.xyz, ray time
    float4 d;     // direction.xyz, t of the pending hit
    float4 a;     // attenuation A.rgb (main.cu:40,51), as_float(prim of the pending hit)
    uint4 ids;    // pixel, sample, bounce (= traces done), leaf texture of the pending hit
};

struct WfBuffers {
    WfRecord* rec;               // [pool]
    uint32_t* queue;             // [2][NQ][pool]
    uint32_t* counts;            // [3][NQ] queue sizes, rotating: cur / next / being-zeroed
    uint32_t* tickets;           // [3] chunk ticket counters, same rotation
    unsigned long long* next_path; // [2], rotating: [it & 1] = paths started before iteration `it`
    uint2* next_ps;                // [2], same rotation: (next_path % pixels, next_path / pixels), kept by the kernels so that
                                   // no thread divides a 64-bit path number (PathMap)
    uint32_t pool;
    // Thin end of a frame (k_wf_tail): once no path is left to start and at most `tail_paths` are alive, the step kernel
    // that sees it records its iteration and the queue sizes in tail[0], tail[1 + q] and leaves; k_wf_tail finishes
    // those paths in place.  tail_paths = 0: never.
    uint32_t tail_paths;
    uint32_t* tail; // [2 + NQ]: iteration (WF_TAIL_NONE: not armed), queue sizes, CTAs of k_wf_tail that have finished
};
#define WF_TAIL_NONE 0xffffffffu

// Where the new paths of an iteration start: entry idx of Q_NEW is path next_path + idx, i.e. pixel
// (pix_base + idx) % npix of sample smp_base + (pix_base + idx) / npix — one 32-bit division by an invariant
// (FastDiv; pix_base < npix < 2^31 and idx < pool <= 2^28 cannot overflow).  n_valid: entries that still get a path.
struct PathMap {
    uint32_t pix_base, smp_base, n_valid;
};
RT_DEV PathMap make_pathmap(const WfBuffers& wb, int it, unsigned long long path_base, uint32_t n_new, unsigned long long npaths) {
    const uint2 ps = wb.next_ps[it & 1];
    const unsigned long long left = npaths > path_base ? npaths - path_base : 0ull;
    return PathMap{ps.x, ps.y, left < n_new ? uint32_t(left) : n_new};
}
// block 0 / thread 0 of every step kernel: the counters of the next iteration
RT_DEV void wf_advance_paths(const WfBuffers& wb, int it, unsigned long long path_base, uint32_t n_new, unsigned long long npix) {
    const unsigned long long next = path_base + n_new;
    wb.next_path[(it + 1) & 1] = next;
    wb.next_ps[(it + 1) & 1] = make_uint2(uint32_t(next % npix), uint32_t(next / npix));
}

struct WavefrontState {
    WfBuffers b{};
    unsigned long long* h_status = nullptr; // pinned [2]: paths started, one per polling parity
    uint32_t* h_counts = nullptr;           // pinned [2][3 * NQ]: queue sizes, one copy per polling parity
    cudaEvent_t poll_ev[2] = {nullptr, nullptr};
    cudaStream_t stream = nullptr;
    bool persist_set = false;
    int persist_max = -1, window_max = 0, l2_bytes = 0; // L2 size and persistence limits of this state's device, queried on first use
};

// Streaming accesses to data that is read once and written once per iteration (path records, queue entries): L1
// evict-first loads and stores (ld/st.global.cs), so they do not displace the stack frames and the sphere data
// (C1 -1.5 %, C2 -1.9 % on the probes, C2 bench -11 % (round-1 A/Bs, logs not kept); L2-only .cg accesses were
// 3.7 % SLOWER than .cs on C1 in round 1).  Used by the CTA-chunk and warp-chunk kernels.
// The persistent-lane kernel uses plain accesses because they keep its image right: with streaming ones its
// million-sphere frame differed from the megakernel's in 0.04 % of the rays, identically for .cs and .cg (so not a
// matter of cache coherence; the kernel sits at its register limit and has shown such a codegen-dependent difference
// once before, DESIGN.md section 3).  The cause is not known, so that kernel keeps the accesses it was verified with.
// k_wf_tail uses plain accesses as well.
enum : int { WF_ACC_PLAIN = 0, WF_ACC_STREAM = 1 };
template <int MODE, typename T>
RT_DEV T wf_ld(const T* p) {
    return MODE == WF_ACC_STREAM ? __ldcs(p) : *p;
}
template <int MODE, typename T>
RT_DEV void wf_st(T* p, T v) {
    if (MODE == WF_ACC_STREAM) __stcs(p, v);
    else *p = v;
}
template <int MODE>
RT_DEV uint32_t wf_qload(const uint32_t* p) {
    return MODE == WF_ACC_STREAM ? __ldcs(p) : __ldg(p);
}
RT_DEV uint32_t* wf_queue(const WfBuffers& b, int parity, int q) { return b.queue + (size_t(parity) * NQ + size_t(q)) * b.pool; }

// Shading class of a hit: material kind x cost class of its (checker-resolved) leaf texture.
// Returns Q_NONE when the path terminates right here (constant emitter): `value` is set.
RT_DEV int classify_hit(const DScene& sc, const DRenderParams& rp, const RayQ& q, Hit h, int32_t& leaf, V3& value) {
    uint32_t mat_ix = __ldg(&sc.sph_c[h.prim]).y;
    float4 m0 = __ldg(reinterpret_cast<const float4*>(sc.mats + mat_ix));
    uint32_t kind = __float_as_uint(m0.x);
    leaf = -1;
    if (kind == RT_MAT_METAL) return Q_METAL;
    if (kind == RT_MAT_DIELECTRIC) return Q_DIEL;
    int32_t tex = __float_as_int(m0.y);
    DTexture t = load_tex(sc, tex);
    leaf = tex;
    if (t.kind == RT_TEX_CHECKER) { // the checker only needs p (texture.h:41-48)
        V3 p = q.o + h.t * q.d;
        leaf = resolve_texture(sc, tex, p, t);
    }
    if (kind == RT_MAT_EMITTER) {
        if (t.kind == RT_TEX_CONSTANT) { // emitter::emit (material.h:50-52) + bloom (main.cu:49)
            float intensity = __ldg(reinterpret_cast<const float4*>(sc.mats + mat_ix) + 1).y;
            value = tex_constant(t) * intensity + mk(rp.bloom, rp.bloom, rp.bloom);
            return Q_NONE;
        }
        return Q_EMIT;
    }
    switch (t.kind) {
    case RT_TEX_CONSTANT: return Q_LAMB_CONST;
    case RT_TEX_NOISE_PERLIN:
    case RT_TEX_WOOD: return Q_LAMB_NOISE1;
    case RT_TEX_NOISE_TURBULANCE:
    case RT_TEX_NOISE_MARBLE: return Q_LAMB_NOISE6;
    case RT_TEX_IMAGE: return Q_LAMB_IMAGE;
    default: return Q_LAMB_CONST;
    }
}

// Per-lane state of one queue entry between its shading step and the end of its ray's traversal.
struct WfLane {
    uint32_t slot, pixel, sample, bounce;
    V3 A;
    Ray r;
    bool nee_vertex;      // NEE instantiations: ln.r leaves a lambertian hit that traced its shadow/emission ray
    uint32_t shadow_rays; // ... and how many such rays wf_begin traced (0 or 1)
};

// First half of one queue entry: shade the pending hit of `slot` (or generate the camera ray of path `path`) and
// scatter.  Returns true when a new ray (ln.r) has to be extended.  Otherwise the entry is finished here —
// emitter, absorbed ray, depth limit, or no path left — and `out_q` says where the slot goes (Q_NEW / Q_NONE).
// NEE = RT_RENDER_EMITTER_SAMPLING (a separate instantiation: the reference estimator's kernels do not change).
// RM = RM_ADAPT: adaptive sampling, new paths take their pixel from rp.adapt_pixels, values go to the plane of the sample's
// parity.  RM = RM_FRAMES: a frame sequence, new paths look through the camera of their sample's frame and values go to
// that frame's accumulator.  Neither changes the path record: pixel and sample determine both.
template <bool NEE, int STREAM, int RM = RM_PLAIN>
RT_DEV bool wf_begin(const DScene& sc, const DRenderParams& rp, const WfBuffers& wb, const PerlinTab& pt, int kind, bool valid,
                     uint32_t slot, uint32_t idx, const PathMap& pm, float4* __restrict__ accum, WfLane& ln, int& out_q) {
    const V3 bloom = mk(rp.bloom, rp.bloom, rp.bloom);
    const WfRecord* rec = wb.rec + slot;
    bool has_ray = false;   // a ray to extend
    bool finished = false;  // path ended: add `A` to the pixel
    bool slot_free = false; // hand the slot to Q_NEW
    V3 A = mk(0.f, 0.f, 0.f);
    bool nee_vertex = false;
    uint32_t shadow_rays = 0;
    uint32_t pixel = 0, sample = 0, bounce = 0;
    Ray r;
    r.o = r.d = mk(0.f, 0.f, 0.f);
    r.time = 0.f;

    if (valid) {
        if (kind == Q_NEW) {
            if (idx < pm.n_valid) {
                const uint32_t x = pm.pix_base + idx, q = fastdiv(x, rp.div_npix);
                pixel = x - q * rp.div_npix.d;
                if (RM == RM_ADAPT) pixel = __ldg(rp.adapt_pixels + pixel);
                sample = pm.smp_base + q + uint32_t(rp.sample_offset);
                A = mk(rp.world_r, rp.world_g, rp.world_b);
                if (rp.max_depth > 0) {
                    r = camera_ray<RM>(sc, rp, pixel, sample);
                    has_ray = true;
                } else { // exceeded recursion before the first hit test (main.cu:42,70)
                    A = mk(0.f, 0.f, 0.f);
                    finished = true;
                    slot_free = true;
                }
            } // else: no paths left; the slot retires
        } else {
            const float4 ro = wf_ld<STREAM>(&rec->o), rd = wf_ld<STREAM>(&rec->d), ra = wf_ld<STREAM>(&rec->a);
            const uint4 ids = wf_ld<STREAM>(&rec->ids);
            pixel = ids.x;
            sample = ids.y;
            bounce = ids.z;
            RayQ q;
            q.o = mk(ro.x, ro.y, ro.z);
            q.d = mk(rd.x, rd.y, rd.z);
            q.time = ro.w;
            q.a = 0.f; // not needed for shading
            Hit h{rd.w, __float_as_uint(ra.w)};
            A = mk(ra.x, ra.y, ra.z);
            V3 p, n;
            hit_surface(sc, q, h, p, n);
            if (kind == Q_EMIT) { // emitter::emit (material.h:50-52): value = tex * intensity + bloom; A is dropped
                DTexture t = load_tex(sc, int32_t(ids.w));
                float intensity = __ldg(reinterpret_cast<const float4*>(sc.mats + __ldg(&sc.sph_c[h.prim]).y) + 1).y;
                A = texture_leaf_value(sc, pt, t, n, p) * intensity + bloom;
                finished = true;
                slot_free = true;
            } else {
                const V3 E = mk(0.f, 0.f, 0.f) + bloom; // material::emit (material.h:14-16) + bloom
                const U4 rn = rng_block(rp.seed, pixel, sample, bounce, 0);
                V3 att;
                bool scattered = true;
                if (kind == Q_METAL) {
                    DMaterial m = load_mat(sc, __ldg(&sc.sph_c[h.prim]).y);
                    att = mk(m.ax, m.ay, m.az);
                    scattered = scatter_metal(q, p, n, m.param, rn, r);
                } else if (kind == Q_DIEL) {
                    DMaterial m = load_mat(sc, __ldg(&sc.sph_c[h.prim]).y);
                    att = mk(m.ax, m.ay, m.az);
                    scatter_dielectric(q, p, n, m.param, rn, r);
                } else {
                    DTexture t = load_tex(sc, int32_t(ids.w));
                    if (kind == Q_LAMB_CONST) att = tex_constant(t);
                    else if (kind == Q_LAMB_NOISE1) att = t.kind == RT_TEX_WOOD ? tex_wood(pt, t, p) : tex_perlin(pt, t, p);
                    else if (kind == Q_LAMB_NOISE6) att = t.kind == RT_TEX_NOISE_MARBLE ? tex_marble(pt, t, p) : tex_turbulence(pt, t, p);
                    else att = tex_image(sc, t, n);
                    scatter_lambertian(q, p, n, rn, r);
                    if (NEE && int(bounce) < rp.max_depth) { // the hit's shadow/emission ray (rt_shade.cuh), traced right here
                        const V3 c = emitter_sample(sc, rp, pt, p, n, q.time, pixel, sample, bounce, shadow_rays);
                        if (c.x != 0.f || c.y != 0.f || c.z != 0.f) atomicAdd(&accum_plane<RM>(accum, rp, sample)[pixel], make_float4(c.x, c.y, c.z, 0.f));
                        nee_vertex = true;
                    }
                }
                if (!scattered) { // absorbed (material.h:129-130): the path's value is E (main.cu:53-54)
                    A = E;
                    finished = true;
                    slot_free = true;
                } else {
                    A = E + att * A; // main.cu:51
                    if (int(bounce) >= rp.max_depth) { // exceeded recursion (main.cu:70)
                        A = mk(0.f, 0.f, 0.f);
                        finished = true;
                        slot_free = true;
                    } else {
                        has_ray = true;
                    }
                }
            }
        }
    }
    if (finished) atomicAdd(&accum_plane<RM>(accum, rp, sample)[pixel], make_float4(A.x, A.y, A.z, 1.f));
    out_q = slot_free ? int(Q_NEW) : Q_NONE;
    ln.nee_vertex = nee_vertex;
    ln.shadow_rays = shadow_rays;
    ln.slot = slot;
    ln.pixel = pixel;
    ln.sample = sample;
    ln.bounce = bounce;
    ln.A = A;
    ln.r = r;
    return has_ray;
}

// Second half: the closest hit `h` of ln.r is known.  Miss / constant emitter: the path ends (accumulate, slot to
// Q_NEW); otherwise the record is stored and the slot goes to the shading queue of the hit.  Returns that queue.
template <bool NEE, int STREAM, int RM = RM_PLAIN>
RT_DEV int wf_finish(const DScene& sc, const DRenderParams& rp, const WfBuffers& wb, float4* __restrict__ accum, WfLane& ln,
                     const RayQ& q, Hit h) {
    WfRecord* rec = wb.rec + ln.slot;
    const uint32_t bounce = ln.bounce + 1u;
    V3 A = ln.A;
    int out_q;
    bool finished = false;
    if (h.prim == RT_INVALID_ID) { // miss: the path's value is A (main.cu:66-67)
        finished = true;
    } else {
        int32_t leaf;
        V3 value;
        out_q = classify_hit(sc, rp, q, h, leaf, value);
        if (NEE && ln.nee_vertex && (out_q == Q_NONE || out_q == Q_EMIT) && light_listed(sc, h.prim)) {
            A = mk(0.f, 0.f, 0.f); // this emitter was counted by the shadow ray of the hit the ray comes from
            finished = true;
        } else if (out_q == Q_NONE) { // constant emitter: terminate here
            A = value;
            finished = true;
        } else {
            wf_st<STREAM>(&rec->o, make_float4(ln.r.o.x, ln.r.o.y, ln.r.o.z, ln.r.time));
            wf_st<STREAM>(&rec->d, make_float4(ln.r.d.x, ln.r.d.y, ln.r.d.z, h.t));
            wf_st<STREAM>(&rec->a, make_float4(A.x, A.y, A.z, __uint_as_float(h.prim)));
            wf_st<STREAM>(&rec->ids, make_uint4(ln.pixel, ln.sample, bounce, uint32_t(leaf)));
        }
    }
    if (finished) {
        atomicAdd(&accum_plane<RM>(accum, rp, ln.sample)[ln.pixel], make_float4(A.x, A.y, A.z, 1.f));
        out_q = Q_NEW;
    }
    return out_q;
}

// One whole queue entry (the CTA-chunk and warp-chunk kernels): begin, closest hit, finish.  Called by all 32 lanes of
// the warp (the BVH traversal is warp-cooperative); `valid` = false for lanes past the end of the queue.
template <bool USE_BVH, bool NEE, int ACC = WF_ACC_STREAM, int LIST = 0, int RM = RM_PLAIN>
RT_DEV int wf_process_entry(const DScene& sc, const DRenderParams& rp, const WfBuffers& wb, const PerlinTab& pt, int kind,
                            bool valid, uint32_t slot, uint32_t idx, const PathMap& pm, float4* __restrict__ accum,
                            unsigned long long& nrays) {
    WfLane ln;
    int out_q;
    const bool has_ray = wf_begin<NEE, ACC, RM>(sc, rp, wb, pt, kind, valid, slot, idx, pm, accum, ln, out_q);
    if (NEE) nrays += ln.shadow_rays;
    if (USE_BVH) {
        const RayQ q = make_rayq(ln.r);
        const Hit h = closest_hit_bvh_warp(sc, q, rp.tmin, has_ray);
        if (has_ray) {
            ++nrays;
            out_q = wf_finish<NEE, ACC, RM>(sc, rp, wb, accum, ln, q, h);
        }
    } else if (has_ray) {
        const RayQ q = make_rayq(ln.r);
        const Hit h = closest_hit_list<LIST>(sc, q, rp.tmin);
        ++nrays;
        out_q = wf_finish<NEE, ACC, RM>(sc, rp, wb, accum, ln, q, h);
    }
    return out_q;
}

// The frame is over when no path is alive and none can start any more; launches the host enqueued ahead of its
// polling then have nothing to do.
// ... or when few enough are alive for k_wf_tail to finish them in place (wb.tail_paths): block 0 then notes the
// iteration and the queue sizes for that kernel (later iterations find empty queues and zero this one's counters).
RT_DEV bool wf_frame_done(const WfBuffers& wb, const uint32_t* cnt_cur, int it, const uint32_t (&n_q)[NQ], unsigned long long path_base,
                          unsigned long long npaths) {
    uint32_t live = 0;
#pragma unroll
    for (int k = 0; k < NQ; ++k) live += k == Q_NEW ? 0u : n_q[k];
    if (path_base < npaths || live > wb.tail_paths) return false;
    if (live != 0u && blockIdx.x == 0 && threadIdx.x < NQ) {
        wb.tail[1 + threadIdx.x] = __ldg(cnt_cur + threadIdx.x);
        if (threadIdx.x == 0) wb.tail[0] = uint32_t(it);
    }
    return true;
}

// Work granularity, variant 1: a CTA takes WF_CTA_THREADS consecutive entries of ONE queue (chunks are drawn from a
// ticket counter) and aggregates its pushes in shared memory: one global atomic per CTA chunk and target queue, two
// block-wide barriers per chunk.  Best when all rays of a chunk cost the same (brute-force scenes): C1 runs 11 % faster
// this way than with warp chunks, whose atomic traffic (~1 atomic per 3.5 ns and queue counter) saturates the L2
// atomic units.
template <bool USE_BVH, bool NEE, int LIST = 0, int RM = RM_PLAIN>
__global__ void __launch_bounds__(WF_CTA_THREADS, WF_CTA_MINBLOCKS)
    k_wf_step_cta(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp, const __grid_constant__ WfBuffers wb,
              int it, float4* __restrict__ accum, unsigned long long* __restrict__ ray_counter) {
    WF_PDL_PROLOGUE();
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t s_count[2][NQ]; // double-buffered by chunk parity: two barriers per chunk instead of four
    __shared__ uint32_t s_base[2][NQ];
    // The chunk a CTA works on next, located by ONE thread (round 1 had all 128 threads redo the search through the
    // per-queue chunk table after every chunk: 5 % of the kernel's instructions, profiles/r02_c1_instruction_diet.md)
    struct __align__(16) Chunk {
        int kind;               // shading queue, -1: no chunk left
        uint32_t first, n_kind; // first entry of the chunk, entries in the queue
        uint32_t pad;
        const uint32_t* q_in;   // the queue
    };
    __shared__ Chunk s_chunk[2];

    const PerlinTab pt{smem, threadIdx.x & 31u};
    const uint32_t lane = threadIdx.x & 31u;

    const uint32_t* cnt_cur = wb.counts + (it % 3) * NQ;
    uint32_t* cnt_next = wb.counts + ((it + 1) % 3) * NQ;
    if (blockIdx.x == 0 && threadIdx.x < NQ) wb.counts[((it + 2) % 3) * NQ + threadIdx.x] = 0; // next iteration's target
    if (blockIdx.x == 0 && threadIdx.x == 0) wb.tickets[(it + 2) % 3] = 0u;                     // and its ticket counter
    const unsigned long long path_base = wb.next_path[it & 1]; // paths started by earlier iterations
    const int par_cur = it & 1, par_next = par_cur ^ 1;

    uint32_t n_q[NQ], chunk_end[NQ];
    uint32_t total_chunks = 0;
#pragma unroll
    for (int k = 0; k < NQ; ++k) n_q[k] = __ldg(cnt_cur + k);
    // chunk order, most expensive classes first so the long chunks start early:
    // NOISE6, NOISE1, IMAGE, EMIT, DIEL, METAL, LAMB_CONST, NEW
    const int order[NQ] = {Q_LAMB_NOISE6, Q_LAMB_NOISE1, Q_LAMB_IMAGE, Q_EMIT, Q_DIEL, Q_METAL, Q_LAMB_CONST, Q_NEW};
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        total_chunks += (n_q[order[k]] + WF_CTA_THREADS - 1) / WF_CTA_THREADS;
        chunk_end[k] = total_chunks;
    }

    // Tail iterations hold a few hundred live paths: CTAs without a chunk leave before staging anything, and
    // the Perlin table is staged only by CTAs that will run a noise shader (their first chunk is the
    // lowest-numbered one they get, and the noise queues come first; textured emitters may need it too).
    const unsigned long long npix = RM == RM_ADAPT ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    const unsigned long long npaths = npix * (unsigned long long)rp.spp;
    if (blockIdx.x == 0 && threadIdx.x == 0) wf_advance_paths(wb, it, path_base, n_q[Q_NEW], npix);
    if (blockIdx.x >= total_chunks) return;
    if (wf_frame_done(wb, cnt_cur, it, n_q, path_base, npaths)) return;
    const PathMap pm = make_pathmap(wb, it, path_base, n_q[Q_NEW], npaths);
    if (sc.has_noise && (blockIdx.x < chunk_end[1] || n_q[Q_EMIT] != 0u)) perlin_stage(smem, threadIdx.x, blockDim.x);
    if (threadIdx.x < 2 * NQ) (&s_count[0][0])[threadIdx.x] = 0u;

    // chunk number -> s_chunk[par] (thread 0 only)
    auto locate = [&](uint32_t chunk, uint32_t par) {
        Chunk c;
        c.kind = -1;
        c.first = c.n_kind = c.pad = 0u;
        c.q_in = nullptr;
        if (chunk < total_chunks) {
            int kpos = 0;
#pragma unroll
            for (int k = 0; k < NQ - 1; ++k) kpos += (chunk >= chunk_end[k]) ? 1 : 0;
            c.kind = order[kpos];
            c.first = (chunk - (kpos ? chunk_end[kpos - 1] : 0u)) * WF_CTA_THREADS;
            c.n_kind = n_q[c.kind];
            c.q_in = wf_queue(wb, par_cur, c.kind);
        }
        s_chunk[par] = c;
    };
    if (threadIdx.x == 0) locate(blockIdx.x, 0u); // the first gridDim.x chunks are implicit: chunk = blockIdx.x
    __syncthreads();

    unsigned long long nrays = 0;
    uint32_t cpar = 0;
    // Chunks are drawn from a ticket counter, so a CTA that got cheap chunks simply takes more of them (against handing
    // chunks out by stride: C1 9.46 -> 9.05 ms per frame).  Thread 0 draws the ticket of the NEXT chunk at the top of a
    // trip and turns it into a chunk record at the bottom — the atomic's latency hides behind the chunk's shading —;
    // the two barriers of the trip publish the record.
    uint32_t* ticket = wb.tickets + (it % 3);
    Chunk ck = s_chunk[0];
    uint32_t slot = (ck.first + threadIdx.x < ck.n_kind) ? wf_qload<WF_ACC_STREAM>(ck.q_in + ck.first + threadIdx.x) : 0u;
    while (ck.kind >= 0) {
        uint32_t drawn = 0u;
        if (threadIdx.x == 0) drawn = atomicAdd(ticket, 1u);
        const uint32_t idx = ck.first + threadIdx.x;
        const bool valid = idx < ck.n_kind;

        const int out_q = wf_process_entry<USE_BVH, NEE, WF_ACC_STREAM, LIST, RM>(sc, rp, wb, pt, ck.kind, valid, slot, idx, pm, accum, nrays);

        // ---- queue push: warp ballot -> shared counters -> one global atomic per queue ----
        uint32_t local = 0;
        {
            const unsigned peers = __match_any_sync(0xffffffffu, out_q);
            if (out_q != Q_NONE) {
                const int leader = __ffs(peers) - 1;
                uint32_t base = 0;
                if (int(lane) == leader) base = atomicAdd(&s_count[cpar][out_q], uint32_t(__popc(peers)));
                base = __shfl_sync(peers, base, leader);
                local = base + uint32_t(__popc(peers & ((1u << lane) - 1u)));
            }
        }
        if (threadIdx.x == 0) locate(gridDim.x + drawn, cpar ^ 1u);
        __syncthreads();
        if (threadIdx.x < NQ) {
            uint32_t c = s_count[cpar][threadIdx.x];
            s_base[cpar][threadIdx.x] = c ? atomicAdd(cnt_next + threadIdx.x, c) : 0u;
            s_count[cpar ^ 1u][threadIdx.x] = 0u; // the other buffer was last read before the barrier above
        }
        __syncthreads();
        if (out_q != Q_NONE) wf_st<WF_ACC_STREAM>(wf_queue(wb, par_next, out_q) + s_base[cpar][out_q] + local, slot);
        cpar ^= 1u;
        // (requesting the next chunk's slot indices a chunk ahead, and prefetching their records, was measured in
        // round 1: 2.6 % and 1.2 % slower with 16 Mi slots)
        ck = s_chunk[cpar]; // written before the two barriers of this trip; rewritten after the first barrier of the next
        if (ck.kind >= 0) slot = ck.first + threadIdx.x < ck.n_kind ? wf_qload<WF_ACC_STREAM>(ck.q_in + ck.first + threadIdx.x) : 0u;
    }

    for (int off = 16; off > 0; off >>= 1) nrays += __shfl_down_sync(0xffffffffu, nrays, off);
    if (lane == 0 && nrays) atomicAdd(ray_counter, nrays);
}


// The thin end of a frame: a CTA-LOCAL wavefront.  Once no path is left to start and few are alive, handing them from
// launch to launch costs a launch per bounce (C1: 58 of 70 iterations carried fewer paths than one wave of threads),
// and nothing a path does from here on concerns another CTA: no path starts, slots retire.  So every CTA takes a share
// of the live paths and runs them to their end on its own: bounce by bounce it regroups its slots by shading class in
// shared memory (class segments padded to whole warps, so a warp still runs one shader with full lanes), processes them
// with the step kernels' entry code (wf_process_entry: shade, scatter, extend, classify; the record carries the path
// between bounces exactly as between two iterations), and block barriers are the only synchronisation.  The first form
// of this kernel gave every path ONE thread for the rest of its life: ncu showed 6.9 of 32 lanes active and 18 times the
// warp instructions of a coherent run (profiles/r02_tail_kernel.md) — the classes of a warp's paths diverge after one bounce.
// A separate kernel, not a loop inside the step kernels: that form cost the bulk 0.8 ms through code generation
// (profiles/r02_c1_instruction_diet.md, section 5).  Launched after every batch of step launches; does nothing until a
// step kernel has set wb.tail[0] (wf_frame_done).
#ifndef WF_TAIL_CAP
#define WF_TAIL_CAP 1280u // slots a CTA can hold, class padding (7 x 31) included
#endif
#ifndef WF_TAIL_THREADS
#define WF_TAIL_THREADS 512 // CTA size of k_wf_tail; one wave of (1024 / WF_TAIL_THREADS) CTAs per SM at 64 registers.  Fewer, larger CTAs keep the
                            // class segments of a CTA dense: 128 x 8 per SM ran at 13 of 32 lanes (profiles/r02_c1_tail_ncu.md); 512 x 2: C2 probe -1.2 %, C3 probe -3 %
#endif
#define WF_TAIL_MINBLOCKS (1024 / WF_TAIL_THREADS)
#define WF_TAIL_DEAD 0xffffffffu
template <bool USE_BVH, bool NEE, int LIST = 0, int RM = RM_PLAIN>
__global__ void __launch_bounds__(WF_TAIL_THREADS, WF_TAIL_MINBLOCKS)
    k_wf_tail(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp, const __grid_constant__ WfBuffers wb,
              float4* __restrict__ accum, unsigned long long* __restrict__ ray_counter) {
    WF_PDL_PROLOGUE();
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t s_in[WF_TAIL_CAP];  // slots grouped by class, class segments start at multiples of 32
    __shared__ uint32_t s_out[WF_TAIL_CAP]; // slot | class << 28 of the paths that go on, WF_TAIL_DEAD for the others
    __shared__ uint32_t s_cnt[NQ], s_cin[NQ], s_off[NQ + 1], s_cur[NQ];
    const uint32_t it = wb.tail[0];
    if (it == WF_TAIL_NONE) return;
    const PerlinTab pt{smem, threadIdx.x & 31u};
    if (sc.has_noise) perlin_stage(smem, threadIdx.x, blockDim.x);
    if (threadIdx.x < NQ) s_cnt[threadIdx.x] = 0u;
    __syncthreads();

    // this CTA's share [lo, hi) of the armed queues, concatenated in shading-cost order
    const int order[NQ - 1] = {Q_LAMB_NOISE6, Q_LAMB_NOISE1, Q_LAMB_IMAGE, Q_EMIT, Q_DIEL, Q_METAL, Q_LAMB_CONST};
    uint32_t total = 0;
#pragma unroll
    for (int k = 0; k < NQ - 1; ++k) total += wb.tail[1 + order[k]];
    const uint32_t per = (total + gridDim.x - 1u) / gridDim.x;
    const uint32_t lo = min(blockIdx.x * per, total), hi = min(lo + per, total);
    uint32_t n_out = hi - lo; // entries of s_out in use
    for (uint32_t i = threadIdx.x; i < n_out; i += blockDim.x) {
        uint32_t idx = lo + i;
        int kind = Q_NONE;
#pragma unroll
        for (int k = 0; k < NQ - 1; ++k) {
            const uint32_t n = wb.tail[1 + order[k]];
            if (kind == Q_NONE) {
                if (idx < n) kind = order[k];
                else idx -= n;
            }
        }
        const uint32_t slot = __ldg(wf_queue(wb, int(it & 1u), kind) + idx);
        s_out[i] = slot | uint32_t(kind) << 28;
        atomicAdd(&s_cnt[kind], 1u);
    }
    const PathMap pm{0u, 0u, 0u}; // no path left to start
    unsigned long long nrays = 0;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) { // class segments of the next bounce, each starting at a multiple of 32
            uint32_t o = 0;
            for (int k = 0; k < NQ; ++k) {
                s_off[k] = o;
                s_cur[k] = 0u;
                s_cin[k] = s_cnt[k];
                o += (s_cnt[k] + 31u) & ~31u;
                s_cnt[k] = 0u;
            }
            s_off[NQ] = o;
        }
        __syncthreads();
        const uint32_t n_in = s_off[NQ];
        if (n_in == 0u) break;
        for (uint32_t i = threadIdx.x; i < n_out; i += blockDim.x) {
            const uint32_t e = s_out[i];
            if (e != WF_TAIL_DEAD) s_in[s_off[e >> 28] + atomicAdd(&s_cur[e >> 28], 1u)] = e & 0x0fffffffu;
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_in; i += blockDim.x) { // n_in is a multiple of 32: whole warps take every trip
            int kind = 0;
#pragma unroll
            for (int k = 1; k < NQ; ++k) kind += (i >= s_off[k]) ? 1 : 0; // (an empty class has s_off[k] == s_off[k + 1]: skipped)
            const bool valid = i - s_off[kind] < s_cin[kind];
            const uint32_t slot = valid ? s_in[i] : 0u;
            const int out_q = wf_process_entry<USE_BVH, NEE, WF_ACC_PLAIN, LIST, RM>(sc, rp, wb, pt, kind, valid, slot, 0u, pm, accum, nrays);
            const bool live = valid && out_q != Q_NONE && out_q != Q_NEW;
            s_out[i] = live ? (slot | uint32_t(out_q) << 28) : WF_TAIL_DEAD;
            if (live) atomicAdd(&s_cnt[out_q], 1u);
        }
        n_out = n_in;
    }
    for (int off = 16; off > 0; off >>= 1) nrays += __shfl_down_sync(0xffffffffu, nrays, off);
    if ((threadIdx.x & 31u) == 0u && nrays) atomicAdd(ray_counter, nrays);
    // the CTA that finishes last (every CTA has read the flag by then) disarms it: the tail launches that follow do nothing
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(&wb.tail[1 + NQ], 1u) == gridDim.x - 1u) {
        wb.tail[1 + NQ] = 0u;
        wb.tail[0] = WF_TAIL_NONE;
    }
}

// Work granularity, variant 2: a WARP draws WF_WCHUNK consecutive entries of ONE queue (WF_ROUNDS rounds of 32) from a
// ticket counter and pushes its results with one global atomic per target queue.  No block-wide barrier inside the
// loop: a warp whose rays finish early moves on instead of waiting for the slowest BVH traversal of the CTA
// (ncu, C2: 21 % of all stall samples sat on that barrier; C2 runs 14 % faster this way, C3 4 %).
// (The shipped build runs one round.  The rounds loop below stays anyway: written without it, nvcc 12.9 sign-extends
// the target queue of the push instead of zero-extending it, and the kernel's SASS changes.)
#ifndef WF_ROUNDS
#define WF_ROUNDS 1
#endif
#define WF_WCHUNK (32 * WF_ROUNDS)
#ifndef WF_CTA_WAVES
#define WF_CTA_WAVES 1u // CTA-chunk kernel: grid = this many waves of resident CTAs; chunks are ticketed, so one wave is enough
#endif
#ifndef RT_WF_BATCH
#define RT_WF_BATCH 8u // launches enqueued between two looks at the polled queue sizes
#endif
#ifndef RT_WF_TAIL_PATHS_DEFAULT
#define RT_WF_TAIL_PATHS_DEFAULT 131072u // live paths from which k_wf_tail takes over (sweep: profiles/r02_tail_kernel.md)
#endif
#ifndef RT_PT_MIN_SPHERES
#define RT_PT_MIN_SPHERES 4096u // persistent-lane kernel from this many primitives on (measured: see profiles/)
#endif
#ifndef WF_PT_THREADS
#define WF_PT_THREADS 128 // CTA size of the persistent-lane kernel
#endif
#ifndef WF_PT_MINBLOCKS
// 7 CTAs of 128 threads = 28 warps per SM at 72 registers.  The kernel waits on dependent node fetches; measured on the full C4
// frame (profiles/r02_c4_traversal.md section 5): 24 warps (80 registers, no spills) 1 489 Mrays/s, 28 warps 1 545, 32 warps
// (64 registers, 100 bytes of spills) 1 539.
#define WF_PT_MINBLOCKS 7
#endif
#ifndef RT_PT_LEAF_LANES_DEFAULT
#define RT_PT_LEAF_LANES_DEFAULT 1
#endif
#ifndef RT_PT_REFILL_DEFAULT
#define RT_PT_REFILL_DEFAULT 16
#endif

template <bool USE_BVH, bool NEE, int RM = RM_PLAIN>
__global__ void __launch_bounds__(WF_THREADS, WF_MINBLOCKS)
    k_wf_step_warp(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp, const __grid_constant__ WfBuffers wb,
              int it, float4* __restrict__ accum, unsigned long long* __restrict__ ray_counter) {
    WF_PDL_PROLOGUE();
    extern __shared__ __align__(16) uint32_t smem[];

    const PerlinTab pt{smem, threadIdx.x & 31u};
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt_mask = (1u << lane) - 1u;

    const uint32_t* cnt_cur = wb.counts + (it % 3) * NQ;
    uint32_t* cnt_next = wb.counts + ((it + 1) % 3) * NQ;
    if (blockIdx.x == 0 && threadIdx.x < NQ) wb.counts[((it + 2) % 3) * NQ + threadIdx.x] = 0; // next iteration's target
    uint32_t* ticket = wb.tickets + (it % 3); // dynamic chunk distribution: warps draw chunk numbers from here
    if (blockIdx.x == 0 && threadIdx.x == 0) wb.tickets[(it + 2) % 3] = 0u;
    const unsigned long long path_base = wb.next_path[it & 1]; // paths started by earlier iterations
    const int par_cur = it & 1, par_next = par_cur ^ 1;

    uint32_t n_q[NQ], chunk_end[NQ];
    uint32_t total_chunks = 0;
#pragma unroll
    for (int k = 0; k < NQ; ++k) n_q[k] = __ldg(cnt_cur + k);
    // chunk order, most expensive classes first so the long chunks start early:
    // NOISE6, NOISE1, IMAGE, EMIT, DIEL, METAL, LAMB_CONST, NEW
    const int order[NQ] = {Q_LAMB_NOISE6, Q_LAMB_NOISE1, Q_LAMB_IMAGE, Q_EMIT, Q_DIEL, Q_METAL, Q_LAMB_CONST, Q_NEW};
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        total_chunks += (n_q[order[k]] + WF_WCHUNK - 1) / WF_WCHUNK;
        chunk_end[k] = total_chunks;
    }

    // Tail iterations hold a few hundred live paths: CTAs without a chunk leave before staging anything, and
    // the Perlin table is staged only by CTAs that will run a noise shader (their first chunk is the
    // lowest-numbered one they get, and the noise queues come first; textured emitters may need it too).
    const unsigned long long npix = RM == RM_ADAPT ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    const unsigned long long npaths = npix * (unsigned long long)rp.spp;
    if (blockIdx.x == 0 && threadIdx.x == 0) wf_advance_paths(wb, it, path_base, n_q[Q_NEW], npix);
    const uint32_t warps_per_cta = WF_THREADS / 32;
    if (blockIdx.x * warps_per_cta >= total_chunks) return;
    if (wf_frame_done(wb, cnt_cur, it, n_q, path_base, npaths)) return;
    const PathMap pm = make_pathmap(wb, it, path_base, n_q[Q_NEW], npaths);
    if (sc.has_noise && (chunk_end[1] != 0u || n_q[Q_EMIT] != 0u)) perlin_stage(smem, threadIdx.x, blockDim.x);
    __syncthreads(); // the only block-wide barrier of the kernel

    unsigned long long nrays = 0;

    // Chunks are handed out dynamically (heavy classes first) so no warp idles at the end of the launch; the
    // ticket for the NEXT chunk is drawn before the current one is processed, which hides the atomic's latency.
    auto draw = [&]() -> uint32_t {
        uint32_t c = 0u;
        if (lane == 0u) c = atomicAdd(ticket, 1u);
        return c;
    };
    uint32_t ticket_next = draw();
    for (;;) {
        const uint32_t chunk = __shfl_sync(0xffffffffu, ticket_next, 0);
        if (chunk >= total_chunks) break;
        ticket_next = draw();
        int kpos = 0;
#pragma unroll
        for (int k = 0; k < NQ - 1; ++k) kpos += (chunk >= chunk_end[k]) ? 1 : 0;
        const int kind = order[kpos];
        const uint32_t first = (chunk - (kpos ? chunk_end[kpos - 1] : 0u)) * WF_WCHUNK;
        const uint32_t n_kind = n_q[kind];
        const uint32_t* q_in = wf_queue(wb, par_cur, kind);

        uint32_t outq_pack = 0u; // 4 bits per round: target queue + 1 (0 = none)

#pragma unroll 1
        for (int e = 0; e < WF_ROUNDS; ++e) {
            const uint32_t idx = first + uint32_t(e) * 32u + lane;
            const bool valid = idx < n_kind;
            const uint32_t slot = valid ? wf_qload<WF_ACC_STREAM>(q_in + idx) : 0u;
            const int out_q = wf_process_entry<USE_BVH, NEE, WF_ACC_STREAM, 0, RM>(sc, rp, wb, pt, kind, valid, slot, idx, pm, accum, nrays);
                outq_pack |= uint32_t(out_q + 1) << (4 * e);
        }

        // ---- queue push: ballots over all rounds -> ONE global atomic per target queue and warp chunk ----
        // lane q (< NQ) owns queue q: it sums the warp's pushes to q, reserves the range, and hands the base out.
        uint32_t my_total = 0u;
        uint32_t rank_r[WF_ROUNDS];
#pragma unroll
        for (int e = 0; e < WF_ROUNDS; ++e) rank_r[e] = 0u;
#pragma unroll
        for (int qk = 0; qk < NQ; ++qk) {
            uint32_t run = 0u;
#pragma unroll
            for (int e = 0; e < WF_ROUNDS; ++e) {
                const bool mine = ((outq_pack >> (4 * e)) & 15u) == uint32_t(qk + 1);
                const unsigned b = __ballot_sync(0xffffffffu, mine);
                if (mine) rank_r[e] = run + uint32_t(__popc(b & lt_mask));
                run += uint32_t(__popc(b));
            }
            if (int(lane) == qk) my_total = run;
        }
        uint32_t my_base = 0u;
        if (lane < uint32_t(NQ) && my_total) my_base = atomicAdd(cnt_next + lane, my_total);
#pragma unroll
        for (int e = 0; e < WF_ROUNDS; ++e) {
            const uint32_t oq1 = (outq_pack >> (4 * e)) & 15u; // queue + 1
            const uint32_t base = __shfl_sync(0xffffffffu, my_base, int(oq1 + 31u) & 31);
            if (oq1) { // the slot index is re-read from the input queue (an L1 hit) instead of living in a register
                const uint32_t slot = wf_qload<WF_ACC_STREAM>(q_in + first + uint32_t(e) * 32u + lane);
                wf_st<WF_ACC_STREAM>(wf_queue(wb, par_next, int(oq1) - 1) + base + rank_r[e], slot);
            }
        }
    }

    for (int off = 16; off > 0; off >>= 1) nrays += __shfl_down_sync(0xffffffffu, nrays, off);
    if (lane == 0 && nrays) atomicAdd(ray_counter, nrays);
}

// Work granularity, variant 3: persistent lanes.  A warp keeps a cursor into its current 32-entry chunk; a lane
// whose ray has finished runs the second half of its entry (classify, store, push) and takes the NEXT entry of
// the cursor — shade, scatter, start the new traversal — while the other lanes keep their half-walked rays.
// The traversal loop is left whenever `refill` lanes are idle, and inside it every lane takes one step per
// iteration — an inner node, or the leaf it stands at — instead of waiting for the warp at every leaf.
// Measured on C4 (1 M spheres, 1920x1080x4, Mrays/s): per-lane while-while in warp chunks 722 (ncu: 5 of 32
// lanes active per instruction, profiles/r01_wavefront_c4_lbvh_ncu.md), speculative rounds in warp chunks
// 775-820 (11 of 32), this kernel 880-940.  On C2/C3 (a few hundred spheres, shading a third of the work) the
// partial-width shading of refilled lanes costs more than the traversal gains (C2: 10.3 -> 7.1 Grays/s), so the
// kernel is used from RT_PT_MIN_SPHERES primitives on.
template <bool NEE, bool QUANT, int RM = RM_PLAIN>
__global__ void __launch_bounds__(WF_PT_THREADS, WF_PT_MINBLOCKS)
    k_wf_step_pt(const __grid_constant__ DScene sc, const __grid_constant__ DRenderParams rp, const __grid_constant__ WfBuffers wb,
                 int it, float4* __restrict__ accum, unsigned long long* __restrict__ ray_counter, int refill, int leaf_lanes) {
    WF_PDL_PROLOGUE();
    extern __shared__ __align__(16) uint32_t smem[];
    __shared__ uint32_t s_nq[NQ], s_cend[NQ];

    const PerlinTab pt{smem, threadIdx.x & 31u};
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lt_mask = (1u << lane) - 1u;

    const uint32_t* cnt_cur = wb.counts + (it % 3) * NQ;
    uint32_t* cnt_next = wb.counts + ((it + 1) % 3) * NQ;
    if (blockIdx.x == 0 && threadIdx.x < NQ) wb.counts[((it + 2) % 3) * NQ + threadIdx.x] = 0; // next iteration's target
    uint32_t* ticket = wb.tickets + (it % 3);
    if (blockIdx.x == 0 && threadIdx.x == 0) wb.tickets[(it + 2) % 3] = 0u;
    const unsigned long long path_base = wb.next_path[it & 1];
    const int par_cur = it & 1, par_next = par_cur ^ 1;

    // chunk order, most expensive classes first: NOISE6, NOISE1, IMAGE, EMIT, DIEL, METAL, LAMB_CONST, NEW
    const int order[NQ] = {Q_LAMB_NOISE6, Q_LAMB_NOISE1, Q_LAMB_IMAGE, Q_EMIT, Q_DIEL, Q_METAL, Q_LAMB_CONST, Q_NEW};
    uint32_t total_chunks = 0, noise_chunks = 0, n_emit = 0, n_new = 0;
#pragma unroll
    for (int k = 0; k < NQ; ++k) {
        const uint32_t n = __ldg(cnt_cur + order[k]);
        total_chunks += (n + 31u) / 32u;
        if (threadIdx.x == 0) {
            s_nq[k] = n;
            s_cend[k] = total_chunks;
        }
        if (k == 1) noise_chunks = total_chunks;
        if (order[k] == Q_EMIT) n_emit = n;
        if (order[k] == Q_NEW) n_new = n;
    }
    const unsigned long long npix = RM == RM_ADAPT ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    const unsigned long long npaths = npix * (unsigned long long)rp.spp;
    if (blockIdx.x == 0 && threadIdx.x == 0) wf_advance_paths(wb, it, path_base, n_new, npix);
    if (blockIdx.x * (WF_PT_THREADS / 32) >= total_chunks) return;
    const PathMap pm = make_pathmap(wb, it, path_base, n_new, npaths);
    if (sc.has_noise && (noise_chunks != 0u || n_emit != 0u)) perlin_stage(smem, threadIdx.x, blockDim.x);
    __syncthreads(); // the only block-wide barrier of the kernel

    unsigned long long nrays = 0;

    auto draw = [&]() -> uint32_t {
        uint32_t c = 0u;
        if (lane == 0u) c = atomicAdd(ticket, 1u);
        return c;
    };
    // warp-aggregated push: one global atomic per target queue
    auto push = [&](int out_q, uint32_t slot) {
        const unsigned peers = __match_any_sync(0xffffffffu, out_q);
        if (out_q != Q_NONE) {
            const int leader = __ffs(peers) - 1;
            uint32_t base = 0u;
            if (int(lane) == leader) base = atomicAdd(cnt_next + out_q, uint32_t(__popc(peers)));
            base = __shfl_sync(peers, base, leader);
            wf_st<WF_ACC_PLAIN>(wf_queue(wb, par_next, out_q) + base + uint32_t(__popc(peers & lt_mask)), slot);
        }
    };

    int stack[RT_BVH4_STACK];
    Trav t;
    t.node = RT_TRAV_DONE;
    t.leaf = 0;
    t.sp = 0;
    t.best = Hit{FLT_MAX, RT_INVALID_ID};
    t.inv = t.noi = mk(0.f, 0.f, 0.f);
    t.e = 0.f;
    RayQ q;
    q.o = q.d = mk(0.f, 0.f, 0.f);
    q.time = q.a = 0.f;
    WfLane ln;
    ln.slot = 0u;
    bool tracing = false; // the lane holds a ray (being traversed, or finished and not yet written back)

    // cursor into the warp's current chunk (warp-uniform)
    int kind = Q_NEW;
    uint32_t pos = 0u, end = 0u;
    const uint32_t* q_in = wb.queue;
    bool more = true;
    uint32_t ticket_next = draw();

    for (;;) {
        // ---- 1. second half of the entries whose ray is done ----
        {
            int out_q = Q_NONE;
            if (tracing && t.node == RT_TRAV_DONE) {
                ++nrays;
                out_q = wf_finish<NEE, WF_ACC_PLAIN, RM>(sc, rp, wb, accum, ln, q, t.best);
                tracing = false;
            }
            push(out_q, ln.slot);
        }
        // ---- 2. idle lanes take the next entries of the cursor ----
        unsigned idle = __ballot_sync(0xffffffffu, !tracing);
        while (idle != 0u && more) {
            if (pos == end) {
                const uint32_t chunk = __shfl_sync(0xffffffffu, ticket_next, 0);
                if (chunk >= total_chunks) {
                    more = false;
                    break;
                }
                ticket_next = draw();
                int kpos = 0;
#pragma unroll
                for (int k = 0; k < NQ - 1; ++k) kpos += (chunk >= s_cend[k]) ? 1 : 0;
                kind = order[kpos];
                pos = (chunk - (kpos ? s_cend[kpos - 1] : 0u)) * 32u;
                end = min(pos + 32u, s_nq[kpos]);
                q_in = wf_queue(wb, par_cur, kind);
            }
            const uint32_t navail = end - pos;
            const uint32_t rank = uint32_t(__popc(idle & lt_mask));
            int out_q = Q_NONE;
            if (!tracing && rank < navail) {
                const uint32_t idx = pos + rank;
                const uint32_t slot = wf_qload<WF_ACC_PLAIN>(q_in + idx);
                if (wf_begin<NEE, WF_ACC_PLAIN, RM>(sc, rp, wb, pt, kind, true, slot, idx, pm, accum, ln, out_q)) {
                    q = make_rayq(ln.r);
                    trav_begin(sc, q, t);
                    t.node = int(sc.root4); // this kernel walks the 4-wide nodes
                    tracing = true;
                }
                if (NEE) nrays += ln.shadow_rays;
            }
            push(out_q, ln.slot);
            pos += min(uint32_t(__popc(idle)), navail);
            idle = __ballot_sync(0xffffffffu, !tracing);
        }
        const unsigned live = __ballot_sync(0xffffffffu, tracing);
        if (live == 0u) break;
        // ---- 3. traverse until `refill` lanes are idle (or, with no work left to hand out, until all are done) ----
        const int keep = more ? max(__popc(live) - refill, 0) : 0;
        int nlive;
        do {
            // One inner-node step for every lane that stands at an inner node; lanes that stand at a leaf (or just
            // arrived at one) test it once `leaf_lanes` of them wait, or when no lane can take an inner step.
            if (t.node >= 0 && t.node != RT_TRAV_DONE) { // 4-wide nodes, 64-byte (quantised) or 128-byte form
                if (QUANT) trav_inner_q(sc, q, rp.tmin, t, stack);
                else trav_inner4(sc, q, rp.tmin, t, stack);
            }
            const unsigned at_leaf = __ballot_sync(0xffffffffu, t.node < 0);
            const unsigned can_go = __ballot_sync(0xffffffffu, t.node >= 0 && t.node != RT_TRAV_DONE);
            if (__popc(at_leaf) >= leaf_lanes || can_go == 0u) {
                if (t.node < 0) trav_leaf(sc, q, rp.tmin, t, stack);
            }
            nlive = __popc(__ballot_sync(0xffffffffu, t.node != RT_TRAV_DONE));
        } while (nlive > keep);
    }

    for (int off = 16; off > 0; off >>= 1) nrays += __shfl_down_sync(0xffffffffu, nrays, off);
    if (lane == 0 && nrays) atomicAdd(ray_counter, nrays);
}

// fills Q_NEW of iteration 0 with every slot (four entries per thread, one 16-byte store: the queue base is 256-byte aligned)
// and resets the counters
__global__ void __launch_bounds__(256) k_wf_init(const __grid_constant__ WfBuffers wb, uint32_t n_slots) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t* q = wf_queue(wb, 0, Q_NEW);
    const uint32_t first = 4u * i;
    if (first + 3u < n_slots) {
        __stcs(reinterpret_cast<uint4*>(q) + i, make_uint4(first, first + 1u, first + 2u, first + 3u));
    } else {
        for (uint32_t k = first; k < n_slots; ++k) q[k] = k;
    }
    if (i < 3 * NQ) wb.counts[i] = (i == Q_NEW) ? n_slots : 0u;
    if (i < 3) wb.tickets[i] = 0u;
    if (i < 2 + NQ) wb.tail[i] = i == 0 ? WF_TAIL_NONE : 0u;
    if (i == 0) {
        wb.next_path[0] = wb.next_path[1] = 0ull;
        wb.next_ps[0] = wb.next_ps[1] = make_uint2(0u, 0u);
    }
}

WavefrontState* wavefront_create(size_t pool_paths, cudaStream_t st) {
    WavefrontState* ws = new WavefrontState();
    ws->stream = st;
    ws->b.pool = uint32_t(pool_paths);
    // (the pool and its queues — 2 GiB at 16 Mi paths — are allocated by the first frame: ensure_slot_buffers)
    bool ok = cudaMallocHost(&ws->h_status, 2 * sizeof(unsigned long long)) == cudaSuccess;
    ok = ok && cudaMallocHost(&ws->h_counts, 2 * 3 * NQ * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ws->poll_ev[0], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ws->poll_ev[1], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        wavefront_destroy(ws);
        return nullptr;
    }
    return ws;
}

static bool ensure_slot_buffers(WavefrontState* ws) {
    if (ws->b.rec) return true;
    const size_t pool_paths = ws->b.pool;
    bool ok = cudaMalloc(&ws->b.rec, pool_paths * sizeof(WfRecord)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.queue, size_t(2) * NQ * pool_paths * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.counts, 3 * NQ * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.tickets, 3 * sizeof(uint32_t)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.next_path, 2 * sizeof(unsigned long long)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.next_ps, 2 * sizeof(uint2)) == cudaSuccess;
    ok = ok && cudaMalloc(&ws->b.tail, (2 + NQ) * sizeof(uint32_t)) == cudaSuccess;
    return ok;
}

void wavefront_destroy(WavefrontState* ws) {
    if (!ws) return;
    if (ws->b.rec) cudaFree(ws->b.rec);
    if (ws->b.queue) cudaFree(ws->b.queue);
    if (ws->b.counts) cudaFree(ws->b.counts);
    if (ws->b.tickets) cudaFree(ws->b.tickets);
    if (ws->b.next_path) cudaFree(ws->b.next_path);
    if (ws->b.next_ps) cudaFree(ws->b.next_ps);
    if (ws->b.tail) cudaFree(ws->b.tail);
    for (auto& e : ws->poll_ev)
        if (e) cudaEventDestroy(e);
    if (ws->h_status) cudaFreeHost(ws->h_status);
    if (ws->h_counts) cudaFreeHost(ws->h_counts);
    delete ws;
}

size_t wavefront_pool(const WavefrontState* ws) { return ws ? ws->b.pool : 0; }

bool wavefront_render(WavefrontState* ws, const DScene& sc, const DRenderParams& rp, bool use_bvh, float4* accum,
                      unsigned long long* ray_counter, int sm_count, cudaStream_t st, uint32_t* launches,
                      uint32_t* iterations) {
    // adaptive sampling: the pass covers the div_npix.d pixels of rp.adapt_pixels (the ADAPT instantiations); a frame
    // sequence covers every pixel, rp.spp samples each over all its frames (the FRAMES instantiations)
    const bool adapt = rp.adapt_pixels != nullptr;
    const int rm = adapt ? RM_ADAPT : (rp.frame_cams ? RM_FRAMES : RM_PLAIN);
    const unsigned long long npix = adapt ? (unsigned long long)rp.div_npix.d : (unsigned long long)rp.width * rp.height;
    const unsigned long long npaths = npix * (unsigned long long)rp.spp;
    *launches = 0;
    *iterations = 0;
    if (npaths == 0) return true;
    // (every build option keeps the table under the 48 KB a kernel may use without a per-device opt-in attribute)
    static_assert(RT_PERLIN_SMEM_WORDS * sizeof(uint32_t) <= 48u * 1024u, "needs cudaFuncAttributeMaxDynamicSharedMemorySize (per device)");
    // scenes without Perlin textures leave the table out
    const size_t smem = sc.has_noise ? RT_PERLIN_SMEM_WORDS * sizeof(uint32_t) : 0;
    // emitter importance sampling: a scene without emitters renders with the reference estimator's kernels
    const bool nee = (rp.flags & RT_RENDER_EMITTER_SAMPLING) != 0u && sc.n_lights > 0u;
    if (!ensure_slot_buffers(ws)) return false;
    // slots in use: never more than there are paths
    WfBuffers wb = ws->b;
    const uint32_t slots = uint32_t(npaths < wb.pool ? npaths : wb.pool);
    wb.tail_paths = 0u; // set below, once the granularity is known; k_wf_init does not read it
    k_wf_init<<<(slots / 4u + 256u) / 256u, 256, 0, st>>>(wb, slots); // (at least one block: it also resets the counters)
    ++*launches;

    // Granularity: CTA chunks (4x fewer queue atomics) when all rays cost the same — the brute-force list —, warp
    // chunks (barrier-free, ticketed) for BVH scenes, persistent lanes with refill when the BVH is large and the
    // rays' traversal lengths spread widely.  RT_WF_GRAIN=cta|warp|pt overrides; RT_PT_REFILL = idle lanes per refill.
    enum { G_CTA, G_WARP, G_PT };
    int grain = !use_bvh ? G_CTA : (sc.n_spheres >= RT_PT_MIN_SPHERES ? G_PT : G_WARP);
    if (const char* e = getenv("RT_WF_GRAIN")) grain = e[0] == 'w' ? G_WARP : (e[0] == 'p' && use_bvh ? G_PT : (e[0] == 'c' ? G_CTA : grain));
    int refill = RT_PT_REFILL_DEFAULT;
    if (const char* e = getenv("RT_PT_REFILL")) {
        const int v = atoi(e);
        if (v >= 1 && v <= 32) refill = v;
    }
    int leaf_lanes = RT_PT_LEAF_LANES_DEFAULT;
    if (const char* e = getenv("RT_PT_LEAF_LANES")) {
        const int v = atoi(e);
        if (v >= 1 && v <= 32) leaf_lanes = v;
    }
    const bool warp_grain = grain != G_CTA;
    // The thin end of the frame is finished in place by k_wf_tail (CTA- and warp-chunk kernels; the persistent-lane kernel
    // walks other nodes than the per-lane loop and its frames spend nothing in the tail).  RT_WF_TAIL_PATHS overrides, 0 = off.
    const unsigned tail_grid = unsigned(sm_count) * WF_TAIL_MINBLOCKS;           // one wave: every CTA owns its paths to their end
    const uint32_t tail_max = tail_grid * (WF_TAIL_CAP - 7u * 31u - 32u);          // what the CTAs' slot lists can hold
    uint32_t tail_paths = grain == G_PT ? 0u : RT_WF_TAIL_PATHS_DEFAULT;
    if (const char* e = getenv("RT_WF_TAIL_PATHS")) {
        const long v = atol(e);
        if (v >= 0 && grain != G_PT) tail_paths = uint32_t(v < (1l << 24) ? v : (1l << 24));
    }
    if (tail_paths > tail_max) tail_paths = tail_max;
    wb.tail_paths = tail_paths;
    // node form of the persistent-lane kernel: the 64-byte quantised nodes when the scene has them (RT_BVH4=f: the 128-byte ones)
    bool quant = sc.nodes4q != nullptr;
    if (const char* e = getenv("RT_BVH4")) quant = quant && e[0] != 'f';
    unsigned grid;
    if (warp_grain) { // resident CTAs only: work is drawn dynamically
        const unsigned cap = unsigned(sm_count) * (grain == G_PT ? WF_PT_MINBLOCKS : WF_MINBLOCKS);
        const unsigned cta_warps = (grain == G_PT ? WF_PT_THREADS : WF_THREADS) / 32;
        const unsigned need = (slots + WF_WCHUNK * cta_warps - 1) / (WF_WCHUNK * cta_warps) + NQ;
        grid = need < cap ? need : cap;
    } else { // two waves of CTAs, chunks by stride
        const unsigned cap = unsigned(sm_count) * WF_CTA_WAVES * WF_CTA_MINBLOCKS;
        const unsigned need = (slots + WF_CTA_THREADS - 1) / WF_CTA_THREADS + NQ;
        grid = need < cap ? need : cap;
    }

    // L2 residency of the BVH: the path records stream through L2 once per iteration (64 B per slot) and would evict
    // the node array, which every ray re-reads along its walk; an access-policy window marks the nodes persisting.
    bool l2_window = false;
    if (use_bvh && sc.nodes && sc.n_nodes >= RT_PT_MIN_SPHERES && !getenv("RT_NO_L2_PERSIST")) {
        int& persist_max = ws->persist_max; // per state, i.e. per context and device (not per process)
        int& window_max = ws->window_max;
        if (persist_max < 0) {
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&persist_max, cudaDevAttrMaxPersistingL2CacheSize, dev);
            cudaDeviceGetAttribute(&window_max, cudaDevAttrMaxAccessPolicyWindowSize, dev);
            cudaDeviceGetAttribute(&ws->l2_bytes, cudaDevAttrL2CacheSize, dev);
        }
        const bool wide = grain == G_PT;
        size_t bytes = size_t(wide ? sc.n_nodes4 : sc.n_nodes) * (wide ? (quant ? sizeof(BvhNode4Q) : sizeof(BvhNode4)) : sizeof(BvhNode));
        // Only for node arrays that the record stream can actually push out: the 32 MB of quantised nodes of the 1 M-sphere scene
        // stay in the 126 MB L2 on their own, and carving a persisting region out of it costs the sphere data and the records
        // more than it saves (C4 1 546 -> 1 570 Mrays/s without the window, profiles/r02_c4_ab_knobs.log; the 64 MB float nodes
        // of round 1 gained from it).
        const bool worth = bytes > size_t(ws->l2_bytes) / 3u || getenv("RT_L2_PERSIST_ALWAYS");
        if (worth && persist_max > 0 && !ws->persist_set) {
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, size_t(persist_max));
            ws->persist_set = true;
        }
        if (worth && persist_max > 0 && window_max > 0) {
            cudaStreamAttrValue av{};
            if (bytes > size_t(window_max)) bytes = size_t(window_max);
            av.accessPolicyWindow.base_ptr = wide ? (quant ? (void*)sc.nodes4q : (void*)sc.nodes4) : (void*)sc.nodes;
            av.accessPolicyWindow.num_bytes = bytes;
            const float ratio = float(double(persist_max) * 0.9 / double(bytes));
            av.accessPolicyWindow.hitRatio = ratio < 1.f ? ratio : 1.f;
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            l2_window = cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &av) == cudaSuccess;
        }
    }

    // every step launch carries the programmatic-stream-serialization attribute (see WF_PDL_PROLOGUE)
    auto launch_dims = [&](unsigned n_blocks, unsigned n_threads, auto kernel, auto... args) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(n_blocks);
        cfg.blockDim = dim3(n_threads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        cudaLaunchKernelEx(&cfg, kernel, args...);
    };
    auto launch = [&](auto kernel, auto... args) { launch_dims(grid, grain == G_PT ? WF_PT_THREADS : (warp_grain ? WF_THREADS : WF_CTA_THREADS), kernel, args...); };
    uint32_t it = 0;
    auto step = [&](auto rm_tag) {
        constexpr int RM = decltype(rm_tag)::value;
        if (grain == G_PT) {
            if (quant) {
                if (nee) launch(k_wf_step_pt<true, true, RM>, sc, rp, wb, int(it), accum, ray_counter, refill, leaf_lanes);
                else launch(k_wf_step_pt<false, true, RM>, sc, rp, wb, int(it), accum, ray_counter, refill, leaf_lanes);
            } else {
                if (nee) launch(k_wf_step_pt<true, false, RM>, sc, rp, wb, int(it), accum, ray_counter, refill, leaf_lanes);
                else launch(k_wf_step_pt<false, false, RM>, sc, rp, wb, int(it), accum, ray_counter, refill, leaf_lanes);
            }
        } else if (warp_grain) {
            if (nee) {
                if (use_bvh) launch(k_wf_step_warp<true, true, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else launch(k_wf_step_warp<false, true, RM>, sc, rp, wb, int(it), accum, ray_counter);
            } else {
                if (use_bvh) launch(k_wf_step_warp<true, false, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else launch(k_wf_step_warp<false, false, RM>, sc, rp, wb, int(it), accum, ray_counter);
            }
        } else {
            if (nee) {
                if (use_bvh) launch(k_wf_step_cta<true, true, 0, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else if (sc.n_list) launch(k_wf_step_cta<false, true, 1, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else launch(k_wf_step_cta<false, true, 2, RM>, sc, rp, wb, int(it), accum, ray_counter);
            } else {
                if (use_bvh) launch(k_wf_step_cta<true, false, 0, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else if (sc.n_list) launch(k_wf_step_cta<false, false, 1, RM>, sc, rp, wb, int(it), accum, ray_counter);
                else launch(k_wf_step_cta<false, false, 2, RM>, sc, rp, wb, int(it), accum, ray_counter);
            }
        }
    };
    auto enqueue = [&](uint32_t count) {
        for (uint32_t k = 0; k < count; ++k, ++it) {
            if (rm == RM_ADAPT) step(std::integral_constant<int, RM_ADAPT>{});
            else if (rm == RM_FRAMES) step(std::integral_constant<int, RM_FRAMES>{});
            else step(std::integral_constant<int, RM_PLAIN>{});
            ++*launches;
        }
    };
    auto tail = [&](auto rm_tag) {
        constexpr int RM = decltype(rm_tag)::value;
        const unsigned nb = tail_grid, nt = WF_TAIL_THREADS;
        if (nee) {
            if (use_bvh) launch_dims(nb, nt, k_wf_tail<true, true, 0, RM>, sc, rp, wb, accum, ray_counter);
            else if (sc.n_list) launch_dims(nb, nt, k_wf_tail<false, true, 1, RM>, sc, rp, wb, accum, ray_counter);
            else launch_dims(nb, nt, k_wf_tail<false, true, 2, RM>, sc, rp, wb, accum, ray_counter);
        } else {
            if (use_bvh) launch_dims(nb, nt, k_wf_tail<true, false, 0, RM>, sc, rp, wb, accum, ray_counter);
            else if (sc.n_list) launch_dims(nb, nt, k_wf_tail<false, false, 1, RM>, sc, rp, wb, accum, ray_counter);
            else launch_dims(nb, nt, k_wf_tail<false, false, 2, RM>, sc, rp, wb, accum, ray_counter);
        }
    };
    auto enqueue_tail = [&]() {
        if (!tail_paths) return;
        if (rm == RM_ADAPT) tail(std::integral_constant<int, RM_ADAPT>{});
        else if (rm == RM_FRAMES) tail(std::integral_constant<int, RM_FRAMES>{});
        else tail(std::integral_constant<int, RM_PLAIN>{});
        ++*launches;
    };
    // Iterations are enqueued in batches.  After each batch the queue sizes and the path counter are copied to
    // pinned memory; the host looks at the copy of batch k only AFTER batch k+1 has been enqueued, so the GPU
    // never waits for the host.  Once the frame is finished the launches still in flight find empty queues and
    // return immediately (every CTA exits before touching anything).
    struct Polled {
        uint32_t it_after; // iterations enqueued when the snapshot was requested
    } polled[2];
    auto snapshot = [&](int par) {
        cudaMemcpyAsync(ws->h_counts + par * 3 * NQ, wb.counts, 3 * NQ * sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(ws->h_status + par, wb.next_path + (it & 1), sizeof(unsigned long long), cudaMemcpyDeviceToHost, st);
        cudaEventRecord(ws->poll_ev[par], st);
        polled[par].it_after = it;
    };
    // Upper bound of the iteration count: a path advances one bounce per iteration and lives at most max_depth + 2
    // of them (ray-gen, max_depth traces, the shading step that finds the depth exhausted); while unstarted paths
    // remain every slot is busy, so the last path starts before iteration npaths * (max_depth + 2) / slots.
    const unsigned long long generations = (npaths + slots - 1) / slots;
    const unsigned long long max_iters = (generations + 1ull) * ((unsigned long long)rp.max_depth + 2ull) + 64ull;
    bool complete = false;
    enqueue(uint32_t(2ull * generations + 4ull < max_iters ? 2ull * generations + 4ull : max_iters)); // a path lives ~2 iterations
    enqueue_tail();
    snapshot(0);
    int par = 0;
    while (true) {
        enqueue(RT_WF_BATCH);
        enqueue_tail();
        snapshot(par ^ 1);
        if (cudaEventSynchronize(ws->poll_ev[par]) != cudaSuccess) break;
        const uint32_t* c = ws->h_counts + par * 3 * NQ + (polled[par].it_after % 3) * NQ; // queues of the next iteration
        uint64_t live = 0;
        for (int k = 0; k < NQ; ++k)
            if (k != Q_NEW) live += c[k];
        const unsigned long long started = ws->h_status[par];
        if (live == 0 && (started >= npaths || c[Q_NEW] == 0)) {
            complete = true;
            break;
        }
        if (it >= max_iters) break; // a bug, not a long frame (see the bound above): reported, never a silently short frame
        par ^= 1;
    }
    *iterations = it;
    if (l2_window) {
        cudaStreamAttrValue av{};
        av.accessPolicyWindow.num_bytes = 0;
        cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &av);
    }
    return complete;
}

} // namespace rtd
