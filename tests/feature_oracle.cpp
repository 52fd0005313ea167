// tests/feature_oracle.cpp — TEST INFRASTRUCTURE: CPU restatement of the denoiser's feature pass (k_features,
// csrc/rt_denoise.cu) with the product's sampler (sampler 1: Philox camera rays exactly as orc_render(..., sampler = 1)
// draws them).  It is compiled as ONE translation unit with oracle/rt_oracle.cpp, whose camera, closest-hit, texture and
// scatter restatements it calls, so the oracle that pins the reference stays as it is.  Built by tests/test_denoise.py:
//   g++ -std=c++17 -O2 -fPIC -shared -ffp-contract=off tests/feature_oracle.cpp -o libfeature_oracle.so
#include "../oracle/rt_oracle.cpp"

extern "C" {

// out: 2 * width * height * 4 floats, the two planes of rt_render_features_device (include/rt_api.h)
void orc_features(const orc_scene* s, const rt_render_params* rp, int feature_spp, int nthreads, float* out) {
    const int W = rp->width, H = rp->height;
    const size_t npix = size_t(W) * size_t(H);
    if (nthreads < 1) nthreads = 1;
    std::atomic<int> next_row{0};
    auto work = [&]() {
        for (;;) {
            const int j = next_row.fetch_add(1);
            if (j >= H) break;
            for (int i = 0; i < W; ++i) {
                const size_t index = size_t(j) * size_t(W) + size_t(i);
                Sampler sm;
                sm.mode = 1;
                sm.seed = rp->seed;
                sm.pixel = uint32_t(index);
                float nx = 0.f, ny = 0.f, nz = 0.f, dist = 0.f, ar = 0.f, ag = 0.f, ab = 0.f;
                int hits = 0;
                for (int k = 0; k < feature_spp; ++k) {
                    sm.sample = uint32_t(rp->sample_offset + k);
                    const Ray r = camera_ray(*s, sm, i, j, W, H);
                    Hit h;
                    if (!scene_hit(*s, r, rp->tmin, FLT_MAX, 1, h)) {
                        ar += rp->world[0];
                        ag += rp->world[1];
                        ab += rp->world[2];
                        continue;
                    }
                    if (!h.uv_set) sphere_uv(h.n, h.u, h.v); // the product derives u/v from n for every sphere kind
                    const rt_material& m = s->materials[s->spheres[h.prim].material];
                    V3 att = mk(0.f, 0.f, 0.f);
                    if (m.kind == RT_MAT_EMITTER) { // (emit + bloom) - bloom, as the device forms it
                        const V3 e = emit(*s, m, h) + mk(rp->bloom, rp->bloom, rp->bloom);
                        att = mk(e.x - rp->bloom, e.y - rp->bloom, e.z - rp->bloom);
                    } else {
                        Ray next;
                        scatter(*s, m, r, h, sm, 1u, att, next);
                    }
                    ++hits;
                    nx += h.n.x;
                    ny += h.n.y;
                    nz += h.n.z;
                    dist += h.t * sqrtf(r.d.x * r.d.x + r.d.y * r.d.y + r.d.z * r.d.z);
                    ar += att.x;
                    ag += att.y;
                    ab += att.z;
                }
                const float fh = float(hits), fk = float(feature_spp);
                float* f0 = out + 4 * index;
                float* f1 = out + 4 * (npix + index);
                f0[0] = hits ? nx / fh : 0.f;
                f0[1] = hits ? ny / fh : 0.f;
                f0[2] = hits ? nz / fh : 0.f;
                f0[3] = hits ? dist / fh : 0.f;
                f1[0] = ar / fk;
                f1[1] = ag / fk;
                f1[2] = ab / fk;
                f1[3] = fh / fk;
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < nthreads; ++t) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
}

} // extern "C"
