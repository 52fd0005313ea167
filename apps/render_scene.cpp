// apps/render_scene.cpp — the C++ host program that replaces the reference's main() (main.cu:368-512)
// for the render path: builds a scene through the façade (include/rt/scenes.hpp keeps the reference's
// constructor calls), hands the flattened description to the C-ABI, renders, converts with the
// reference's writer loop and stores the frame.
//
//   render_scene [scene] [width height spp] [out] [earth.ppm]            (positional, as before)
//   render_scene --scene <name | file.json> [--width W --height H --spp N --depth D --seed S]
//                [--out render.jpg|.ppm] [--quality 100] [--earth assets/earth_stb.ppm] [--passes K] [--emitter-sampling]
//                [--gpus N] [--denoise] [--adaptive T [--max-spp N]] [--frames N [--orbit DEG]]
//     scene: earth_emitter (default) | book1_final | perlin_motion | random_spheres:N | a JSON document
//            (include/rt/scene_json.hpp; the reference's compile-time scene and WIDTH/HEIGHT/SAMPLES_PER_PIXEL/SEED
//            macros, main.cu:15,188-356, common.h:13-20, become runtime input)
//     out:   *.jpg -> the device output stage (rt_render_jpeg: the same bytes stbi_write_jpg(…, 100) writes,
//            main.cu:491); anything else -> binary PPM of the same pixels
//     --emitter-sampling: RT_RENDER_EMITTER_SAMPLING — lambertian hits aim half of their scatter directions at the
//            emitter spheres and weight the path accordingly (the reference README's "Improve Sampling on emitter
//            objects", README.md:27-28); same expected image, less noise where emitters light the scene
//     --gpus N: N devices from this one process (rt_multi_*; 0 = every visible device): the samples per pixel are split
//            across the devices, the float4 accumulators are summed and finalised by one fused kernel per device over
//            NVLink peer memory.  The output file is written from the 8-bit frame (JPEG through rt_jpeg_encode).
//     --passes K: progressive accumulation, K passes of --spp samples each into one accumulator; the output file is
//            rewritten after every pass (PPM only)
//     --denoise: rt_render_denoised with rt_default_denoise_params — first-hit features and the edge-avoiding à-trous
//            filter on the device after the render; the frame is then written as without it.  One device, one pass.
//     --adaptive T: adaptive sampling (rt_render_adaptive): every pixel gets --spp samples, then passes of --spp samples go
//            to the pixels whose display-space noise estimate is still >= T, up to --max-spp (default 16 x --spp).  With
//            --denoise the adaptive accumulator goes through the device entries (features, rt_denoise_device).  One device.
//     --frames N: a sequence of N frames in one render (rt_render_frames_device): the cameras come from rt_orbit_cameras on
//            the scene's camera, lookfrom turned by --orbit DEG degrees in all (default 0) about the axis through lookat
//            along up, and the shutter split into N windows (so the moving spheres of perlin_motion move from frame to
//            frame).  Frame k is written to <stem>_<kkkk><ext> (render_0000.jpg, ...) through rt_tonemap_device and the
//            device JPEG writer (PPM for other extensions).  One device, one pass, no denoising or adaptive sampling.
//
// The earth texture: --earth textures/earth.jpg (decoded by rt_image_load exactly as stbi_loadf does) or a binary PPM
// of the stb-decoded bytes (assets/earth_stb.ppm, written by __graft_entry__.build()).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../include/rt/scenes.hpp"

#define CHECK(x)                                                                   \
    do {                                                                           \
        rt_status st__ = (x);                                                      \
        if (st__ != RT_OK) {                                                       \
            fprintf(stderr, "%s failed (%d): %s\n", #x, int(st__), rt_last_error()); \
            return 1;                                                              \
        }                                                                          \
    } while (0)

static bool ends_with(const std::string& s, const char* suf) {
    const size_t n = strlen(suf);
    return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

int main(int argc, char** argv) {
    std::string scene_name = "earth_emitter", out_path = "render.jpg", earth_path = "assets/earth_stb.ppm";
    int quality = 100; // main.cu:491
    int passes = 1;
    int gpus = 1; // 1: the single-device path below; anything else: rt_multi_*
    bool emitter_sampling = false;
    bool denoise = false;
    bool adaptive = false;
    float threshold = 0.f;
    int max_spp = 0; // 0: 16 x --spp
    int frames = 0;  // 0: one frame of the scene's camera
    float orbit = 0.f;
    rt_render_params p;
    rt_default_render_params(&p); // 1200x600x100, depth 50, seed 1000, tmin 1e-5 (common.h:13-20, main.cu:15,45)
    bool size_given = false;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto next = [&](const char* what) -> const char* {
            if (i + 1 >= argc) {
                fprintf(stderr, "%s needs a value\n", what);
                exit(2);
            }
            return argv[++i];
        };
        if (a == "--scene") scene_name = next("--scene");
        else if (a == "--width") p.width = atoi(next("--width")), size_given = true;
        else if (a == "--height") p.height = atoi(next("--height")), size_given = true;
        else if (a == "--spp") p.spp = atoi(next("--spp")), size_given = true;
        else if (a == "--depth") p.max_depth = atoi(next("--depth"));
        else if (a == "--seed") p.seed = uint32_t(atoll(next("--seed")));
        else if (a == "--out") out_path = next("--out");
        else if (a == "--quality") quality = atoi(next("--quality"));
        else if (a == "--earth") earth_path = next("--earth");
        else if (a == "--passes") passes = atoi(next("--passes"));
        else if (a == "--gpus") gpus = atoi(next("--gpus"));
        else if (a == "--emitter-sampling") emitter_sampling = true;
        else if (a == "--denoise") denoise = true;
        else if (a == "--adaptive") adaptive = true, threshold = float(atof(next("--adaptive")));
        else if (a == "--max-spp") max_spp = atoi(next("--max-spp"));
        else if (a == "--frames") {
            frames = atoi(next("--frames"));
            if (frames < 1) {
                fprintf(stderr, "--frames needs N >= 1\n");
                return 2;
            }
        } else if (a == "--orbit") orbit = float(atof(next("--orbit")));
        else if (a == "--help" || a == "-h") {
            printf("render_scene --scene <name|file.json> [--width W --height H --spp N --depth D --seed S] [--out f.jpg|f.ppm] "
                   "[--quality Q] [--earth earth.ppm] [--passes K] [--emitter-sampling] [--gpus N] [--denoise] "
                   "[--adaptive T [--max-spp N]] [--frames N [--orbit DEG]]\n");
            return 0;
        } else pos.push_back(a);
    }
    if (pos.size() > 0) scene_name = pos[0];
    if (pos.size() > 3) {
        p.width = atoi(pos[1].c_str());
        p.height = atoi(pos[2].c_str());
        p.spp = atoi(pos[3].c_str());
        size_given = true;
    }
    if (pos.size() > 4) out_path = pos[4];
    if (pos.size() > 5) earth_path = pos[5];
    if (denoise && (gpus != 1 || passes > 1)) {
        fprintf(stderr, "--denoise renders one pass on one device: it cannot be combined with --gpus or --passes\n");
        return 2;
    }
    if (adaptive && (gpus != 1 || passes > 1)) {
        fprintf(stderr, "--adaptive renders on one device and chooses its own passes: it cannot be combined with --gpus or --passes\n");
        return 2;
    }
    if (frames > 0 && (gpus != 1 || passes > 1 || denoise || adaptive)) {
        fprintf(stderr, "--frames renders one pass per frame on one device: it cannot be combined with --gpus, --passes, --denoise or --adaptive\n");
        return 2;
    }

    rt_context* ctx = nullptr;
    CHECK(rt_context_create(0, &ctx));
    rt::arena A;
    rt::scenes::built b;
    float* earth = nullptr;
    rt_scene_desc* json_desc = nullptr;
    if (ends_with(scene_name, ".json")) {
        rt_render_params from_doc = p;
        CHECK(rt_scene_desc_from_json_file(ctx, scene_name.c_str(), &from_doc, &json_desc));
        if (!size_given) p = from_doc; // command-line sizes win over the document's "render" block
        p.flags = from_doc.flags;
    } else if (scene_name == "earth_emitter") {
        int32_t ew = 0, eh = 0;
        // stbi_loadf (main.cu:376-380): a .jpg goes through the JPEG reader (host Huffman + device pixel stages, the same
        // floats stb returns), a .ppm/.pgm is read directly
        CHECK(rt_image_load(ctx, earth_path.c_str(), &earth, &ew, &eh));
        b = rt::scenes::earth_emitter(A, earth, ew, eh);
    } else if (scene_name == "book1_final") {
        b = rt::scenes::book1_final(A);
    } else if (scene_name == "perlin_motion") {
        b = rt::scenes::perlin_motion(A);
    } else if (scene_name.rfind("random_spheres", 0) == 0) {
        uint32_t n = scene_name.size() > 15 ? uint32_t(atoll(scene_name.c_str() + 15)) : 100000u;
        b = rt::scenes::random_spheres(A, n);
    } else {
        fprintf(stderr, "unknown scene %s\n", scene_name.c_str());
        return 2;
    }
    rt::flat_scene fs;
    rt_scene_desc desc;
    if (json_desc) {
        desc = *json_desc;
    } else {
        fs = rt::flatten(*b.list, *b.cam);
        desc = fs.desc();
    }

    if (emitter_sampling) p.flags |= RT_RENDER_EMITTER_SAMPLING;
    if (gpus != 1) { // several devices, one process
        rt_multi* m = nullptr;
        CHECK(rt_multi_create(nullptr, gpus, &m));
        CHECK(rt_multi_set_scene(m, &desc));
        printf("Rendering a %dx%d image (%d samples per pixel) on %d devices\n", p.width, p.height, p.spp, rt_multi_size(m));
        std::vector<uint8_t> img(size_t(p.width) * p.height * 3);
        rt_stats st;
        float ms_reduce = 0.f;
        CHECK(rt_multi_render(m, &p, nullptr, img.data(), &st, &ms_reduce));
        printf("took %.0fus.  (%.1f Mpaths/s, %.1f Mrays/s over %d devices; slowest device %.3f ms, fused reduce + finalisation %.3f ms)\n",
               st.ms_d2h * 1e3, st.paths / st.ms_d2h / 1e3, st.rays / st.ms_d2h / 1e3, rt_multi_size(m), st.ms_total, ms_reduce);
        if (ends_with(out_path, ".jpg") || ends_with(out_path, ".jpeg")) CHECK(rt_write_jpg(ctx, out_path.c_str(), p.width, p.height, img.data(), quality));
        else CHECK(rt_write_ppm(out_path.c_str(), p.width, p.height, img.data()));
        rt_multi_destroy(m);
        rt_context_destroy(ctx);
        rt_free(earth);
        rt_scene_desc_free(json_desc);
        return 0;
    }
    rt_scene* scene = nullptr;
    CHECK(rt_scene_create(ctx, &desc, &scene));
    rt_scene_info info;
    CHECK(rt_scene_get_info(scene, &info));
    printf("Rendering a %dx%d image (%d samples per pixel): %u spheres, %u BVH nodes (mode %u, build %.3f ms)\n", p.width,
           p.height, p.spp, info.n_spheres, info.n_nodes, info.bvh_mode, info.ms_build);

    rt_stats st;
    auto write_frame = [&](const std::vector<float>& fb) -> int {
        std::vector<uint8_t> img(fb.size());
        CHECK(rt_quantize_rgb8(fb.data(), p.width, p.height, img.data())); // main.cu:475-488
        if (ends_with(out_path, ".jpg") || ends_with(out_path, ".jpeg")) CHECK(rt_write_jpg(ctx, out_path.c_str(), p.width, p.height, img.data(), quality));
        else CHECK(rt_write_ppm(out_path.c_str(), p.width, p.height, img.data()));
        return 0;
    };
    if (frames > 0) { // one wavefront for the whole sequence, then per frame: finalisation -> 8-bit frame -> file
        std::vector<rt_camera> cams(frames);
        CHECK(rt_orbit_cameras(&desc.camera, frames, orbit, cams.data()));
        const size_t npix = size_t(p.width) * p.height;
        void *accum = nullptr, *rgb8 = nullptr;
        if (cudaMalloc(&accum, size_t(frames) * npix * 16) != cudaSuccess || cudaMalloc(&rgb8, npix * 3) != cudaSuccess ||
            cudaMemset(accum, 0, size_t(frames) * npix * 16) != cudaSuccess || cudaDeviceSynchronize() != cudaSuccess) {
            fprintf(stderr, "device allocation failed\n");
            return 1;
        }
        CHECK(rt_render_frames_device(ctx, scene, &p, cams.data(), frames, accum, &st));
        printf("took %.0fus for %d frames (%.3f ms per frame; %.1f Mpaths/s, %.1f Mrays/s, %u launches)\n", st.ms_total * 1e3, frames,
               st.ms_total / frames, st.paths / st.ms_total / 1e3, st.rays / st.ms_total / 1e3, st.launches);
        const size_t slash = out_path.find_last_of('/'), dot = out_path.find_last_of('.');
        const bool has_ext = dot != std::string::npos && (slash == std::string::npos || dot > slash);
        const std::string stem = has_ext ? out_path.substr(0, dot) : out_path, ext = has_ext ? out_path.substr(dot) : "";
        const bool jpg = ext == ".jpg" || ext == ".jpeg";
        std::vector<uint8_t> file(jpg ? rt_jpeg_max_bytes(p.width, p.height) : npix * 3);
        for (int k = 0; k < frames; ++k) {
            char num[16];
            snprintf(num, sizeof num, "_%04d", k);
            const std::string path = stem + num + ext;
            CHECK(rt_tonemap_device(ctx, static_cast<char*>(accum) + size_t(k) * npix * 16, p.width, p.height, nullptr, rgb8));
            if (jpg) {
                size_t n = 0;
                CHECK(rt_jpeg_encode_device(ctx, rgb8, p.width, p.height, quality, file.data(), file.size(), &n, nullptr));
                FILE* f = fopen(path.c_str(), "wb");
                const bool ok = f && fwrite(file.data(), 1, n, f) == n;
                if (f) fclose(f);
                if (!ok) {
                    fprintf(stderr, "cannot write %s\n", path.c_str());
                    return 1;
                }
            } else {
                CHECK(rt_context_synchronize(ctx));
                if (cudaMemcpy(file.data(), rgb8, npix * 3, cudaMemcpyDeviceToHost) != cudaSuccess) {
                    fprintf(stderr, "cudaMemcpy failed\n");
                    return 1;
                }
                CHECK(rt_write_ppm(path.c_str(), p.width, p.height, file.data()));
            }
        }
        cudaFree(accum);
        cudaFree(rgb8);
    } else if (adaptive) {
        rt_adaptive_params a;
        rt_default_adaptive_params(&a);
        a.min_spp = a.step_spp = p.spp;
        a.max_spp = max_spp > 0 ? max_spp : 16 * p.spp;
        a.threshold = threshold;
        const size_t npix = size_t(p.width) * p.height;
        std::vector<float> fb(npix * 3);
        int32_t n_passes = 0;
        if (!denoise) {
            std::vector<int32_t> spp_map(npix);
            CHECK(rt_render_adaptive(ctx, scene, &p, &a, fb.data(), spp_map.data(), &st));
            int32_t top = 0;
            for (int32_t c : spp_map) top = c > top ? c : top;
            n_passes = 1 + (top - a.min_spp) / a.step_spp;
        } else { // adaptive accumulator -> first-hit features -> à-trous filter + finalisation, all on the device
            rt_denoise_params d;
            rt_default_denoise_params(&d);
            void *accum = nullptr, *features = nullptr, *rgb = nullptr;
            if (cudaMalloc(&accum, npix * 16) != cudaSuccess || cudaMalloc(&features, 2 * npix * 16) != cudaSuccess ||
                cudaMalloc(&rgb, npix * 3 * sizeof(float)) != cudaSuccess) {
                fprintf(stderr, "cudaMalloc failed\n");
                return 1;
            }
            CHECK(rt_render_adaptive_device(ctx, scene, &p, &a, accum, nullptr, &n_passes, &st));
            CHECK(rt_render_features_device(ctx, scene, &p, d.feature_spp, features));
            CHECK(rt_denoise_device(ctx, accum, features, p.width, p.height, &d, rgb, nullptr));
            CHECK(rt_context_synchronize(ctx));
            if (cudaMemcpy(fb.data(), rgb, fb.size() * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess) {
                fprintf(stderr, "cudaMemcpy failed\n");
                return 1;
            }
            cudaFree(accum);
            cudaFree(features);
            cudaFree(rgb);
        }
        printf("took %.0fus.  (%d passes, mean %.2f samples per pixel of %d..%d, threshold %g; %.1f Mpaths/s, %.1f Mrays/s%s)\n",
               st.ms_total * 1e3, n_passes, double(st.paths) / double(npix), a.min_spp, a.max_spp, double(a.threshold),
               st.paths / st.ms_total / 1e3, st.rays / st.ms_total / 1e3, denoise ? "; denoised" : "");
        if (write_frame(fb)) return 1;
    } else if (passes > 1) { // progressive: the frame on disk sharpens pass by pass
        struct Sink {
            const rt_render_params* p;
            const char* path;
        } sink{&p, out_path.c_str()};
        std::vector<float> fb(size_t(p.width) * p.height * 3);
        auto on_pass = [](int32_t pass, int32_t spp, const float* rgb, void* user) -> int {
            const Sink* s = static_cast<const Sink*>(user);
            std::vector<uint8_t> img(size_t(s->p->width) * s->p->height * 3);
            if (rt_quantize_rgb8(rgb, s->p->width, s->p->height, img.data()) != RT_OK ||
                rt_write_ppm(s->path, s->p->width, s->p->height, img.data()) != RT_OK)
                return 1;
            printf("pass %d: %d samples per pixel written to %s\n", pass, spp, s->path);
            return 0;
        };
        CHECK(rt_render_progressive(ctx, scene, &p, passes, fb.data(), on_pass, &sink, &st));
        printf("took %.0fus on the device for %d passes (%.1f Mpaths/s)\n", st.ms_total * 1e3, passes, st.paths / st.ms_total / 1e3);
    } else if (denoise) {
        std::vector<float> fb(size_t(p.width) * p.height * 3);
        rt_denoise_params d;
        rt_default_denoise_params(&d);
        CHECK(rt_render_denoised(ctx, scene, &p, &d, fb.data(), &st));
        printf("took %.0fus.  (%.1f Mpaths/s, %.1f Mrays/s; features + %d filter levels + finalisation %.3f ms)\n", st.ms_total * 1e3,
               st.paths / st.ms_total / 1e3, st.rays / st.ms_total / 1e3, d.iterations, st.ms_tonemap);
        std::vector<uint8_t> img(fb.size());
        CHECK(rt_quantize_rgb8(fb.data(), p.width, p.height, img.data())); // main.cu:475-488
        if (ends_with(out_path, ".jpg") || ends_with(out_path, ".jpeg")) CHECK(rt_write_jpg(ctx, out_path.c_str(), p.width, p.height, img.data(), quality));
        else CHECK(rt_write_ppm(out_path.c_str(), p.width, p.height, img.data()));
    } else if (ends_with(out_path, ".jpg") || ends_with(out_path, ".jpeg")) {
        // device output stage: finalise, flip, quantise and JPEG-encode on the GPU; only the file comes back
        std::vector<uint8_t> file(rt_jpeg_max_bytes(p.width, p.height));
        size_t n = 0;
        CHECK(rt_render_jpeg(ctx, scene, &p, quality, file.data(), file.size(), &n, &st));
        FILE* f = fopen(out_path.c_str(), "wb");
        if (!f || fwrite(file.data(), 1, n, f) != n) {
            fprintf(stderr, "cannot write %s\n", out_path.c_str());
            return 1;
        }
        fclose(f);
        printf("took %.0fus.  (%.1f Mpaths/s, %.1f Mrays/s, %u launches; JPEG %zu bytes in %.3f ms on the device)\n", st.ms_total * 1e3,
               st.paths / st.ms_total / 1e3, st.rays / st.ms_total / 1e3, st.launches, n, st.ms_d2h);
    } else {
        std::vector<float> fb(size_t(p.width) * p.height * 3);
        CHECK(rt_render(ctx, scene, &p, fb.data(), &st));
        printf("took %.0fus.  (%.1f Mpaths/s, %.1f Mrays/s, %u launches)\n", st.ms_total * 1e3, st.paths / st.ms_total / 1e3,
               st.rays / st.ms_total / 1e3, st.launches);
        std::vector<uint8_t> img(fb.size());
        CHECK(rt_quantize_rgb8(fb.data(), p.width, p.height, img.data())); // main.cu:475-488
        CHECK(rt_write_ppm(out_path.c_str(), p.width, p.height, img.data()));
    }
    rt_scene_destroy(scene);
    rt_context_destroy(ctx);
    rt_free(earth);
    rt_scene_desc_free(json_desc);
    return 0;
}
