// rt_host.cpp — host-only entry points of the C-ABI: built-in scenes (through the
// façade), scene-description files, and the reference's writer conversion.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/rt/scene_json.hpp"
#include "../../include/rt/scenes.hpp"
#include "../../include/rt_api.h"

namespace rtd {
void set_error_message(const char* msg); // rt_api.cu
bool camera_finite(const rt_camera& c); // rt_api.cu
}

namespace {

// rt_scene_desc that owns its arrays; `desc` must stay the first member.
struct OwnedDesc {
    rt_scene_desc desc;
    rt::flat_scene fs;
    std::vector<std::vector<float>> image_data;
    void bind() {
        for (size_t i = 0; i < fs.images.size(); ++i) fs.images[i].rgb = image_data[i].data();
        desc = fs.desc();
    }
};

} // namespace

extern "C" {

size_t rt_abi_sizeof(const char* name) {
    if (!name) return 0;
#define RT_SZ(T) if (strcmp(name, #T) == 0) return sizeof(T)
    RT_SZ(rt_sphere); RT_SZ(rt_material); RT_SZ(rt_texture); RT_SZ(rt_image); RT_SZ(rt_camera); RT_SZ(rt_scene_desc);
    RT_SZ(rt_jpeg_component); RT_SZ(rt_jpeg_coefficients);
    RT_SZ(rt_render_params); RT_SZ(rt_stats); RT_SZ(rt_scene_info); RT_SZ(rt_ray); RT_SZ(rt_hit); RT_SZ(rt_shade_sample);
    RT_SZ(rt_denoise_params); RT_SZ(rt_adaptive_params);
#undef RT_SZ
    return 0;
}

rt_status rt_orbit_cameras(const rt_camera* base, int32_t n_frames, float degrees, rt_camera* out) {
    auto fail = [](const char* msg) {
        rtd::set_error_message((std::string("invalid argument: ") + msg).c_str());
        return RT_ERR_INVALID_ARG;
    };
    if (!base || !out) return fail("base/out is NULL");
    if (n_frames < 1) return fail("n_frames must be >= 1");
    if (!std::isfinite(degrees) || !rtd::camera_finite(*base)) return fail("degrees / camera parameter is not finite");
    const double ux = base->up[0], uy = base->up[1], uz = base->up[2], ul = std::sqrt(ux * ux + uy * uy + uz * uz);
    if (!(ul > 0.0)) return fail("camera up is zero");
    // Rodrigues' rotation of v = lookfrom - lookat about the unit axis a = up / |up|:
    //   v' = v cos(th) + (a x v) sin(th) + a (a . v) (1 - cos(th))
    const double ax = ux / ul, ay = uy / ul, az = uz / ul;
    const double vx = double(base->lookfrom[0]) - base->lookat[0], vy = double(base->lookfrom[1]) - base->lookat[1],
                 vz = double(base->lookfrom[2]) - base->lookat[2];
    const double adv = ax * vx + ay * vy + az * vz;
    const double t0 = base->time0, t1 = base->time1, n = n_frames;
    for (int32_t k = 0; k < n_frames; ++k) {
        const double th = double(degrees) * k / n * (M_PI / 180.0), c = std::cos(th), s = std::sin(th);
        rt_camera cam = *base;
        cam.lookfrom[0] = float(base->lookat[0] + (vx * c + (ay * vz - az * vy) * s + ax * adv * (1.0 - c)));
        cam.lookfrom[1] = float(base->lookat[1] + (vy * c + (az * vx - ax * vz) * s + ay * adv * (1.0 - c)));
        cam.lookfrom[2] = float(base->lookat[2] + (vz * c + (ax * vy - ay * vx) * s + az * adv * (1.0 - c)));
        cam.time0 = float(t0 + (t1 - t0) * k / n);
        cam.time1 = float(t0 + (t1 - t0) * (k + 1) / n);
        out[k] = cam;
    }
    return RT_OK;
}

rt_status rt_quantize_rgb8(const float* rgb, int32_t width, int32_t height, uint8_t* out) {
    if (!rgb || !out || width <= 0 || height <= 0) return RT_ERR_INVALID_ARG;
    // main.cu:476-487
    for (int j = height - 1; j >= 0; --j) {
        for (int i = 0; i < width; ++i) {
            size_t index = size_t(j) * size_t(width) + size_t(i);
            size_t rev_index = size_t(height - j - 1) * size_t(width) + size_t(i);
            out[rev_index * 3 + 0] = uint8_t(int(255.999f * rgb[index * 3 + 0]) & 255);
            out[rev_index * 3 + 1] = uint8_t(int(255.999f * rgb[index * 3 + 1]) & 255);
            out[rev_index * 3 + 2] = uint8_t(int(255.999f * rgb[index * 3 + 2]) & 255);
        }
    }
    return RT_OK;
}

rt_status rt_write_ppm(const char* path, int32_t width, int32_t height, const uint8_t* rgb8) {
    if (!path || !rgb8 || width <= 0 || height <= 0) return RT_ERR_INVALID_ARG;
    FILE* f = fopen(path, "wb");
    if (!f) return RT_ERR_IO;
    fprintf(f, "P6\n%d %d\n255\n", width, height);
    size_t n = size_t(width) * size_t(height) * 3;
    bool ok = fwrite(rgb8, 1, n, f) == n;
    ok = (fclose(f) == 0) && ok;
    return ok ? RT_OK : RT_ERR_IO;
}

// Binary PPM -> float RGB with value = byte/255.f, i.e. what stbi_loadf returns with
// ldr_to_hdr gamma = scale = 1 (main.cu:378-380; stb_image.h:1797-1810).
rt_status rt_read_ppm_f32(const char* path, float** out_rgb, int32_t* width, int32_t* height) {
    if (!path || !out_rgb || !width || !height) return RT_ERR_INVALID_ARG;
    *out_rgb = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return RT_ERR_IO;
    int w = 0, h = 0, maxv = 0;
    char magic[3] = {0, 0, 0};
    auto skip = [&]() {
        int c;
        while ((c = fgetc(f)) != EOF) {
            if (c == '#') {
                while ((c = fgetc(f)) != EOF && c != '\n') {}
            } else if (c != ' ' && c != '\n' && c != '\r' && c != '\t') {
                ungetc(c, f);
                break;
            }
        }
    };
    bool ok = fread(magic, 1, 2, f) == 2 && magic[0] == 'P' && (magic[1] == '6' || magic[1] == '5'); // P5: one channel
    const int ch = magic[1] == '5' ? 1 : 3;
    if (ok) { skip(); ok = fscanf(f, "%d", &w) == 1; }
    if (ok) { skip(); ok = fscanf(f, "%d", &h) == 1; }
    if (ok) { skip(); ok = fscanf(f, "%d", &maxv) == 1; }
    ok = ok && w > 0 && h > 0 && maxv == 255 && fgetc(f) != EOF;
    if (!ok) {
        fclose(f);
        return RT_ERR_IO;
    }
    // the header of a damaged file must not size an allocation: the pixel bytes have to be there
    const long data_at = ftell(f);
    uint64_t left = 0;
    if (data_at >= 0 && fseek(f, 0, SEEK_END) == 0) {
        const long end = ftell(f);
        if (end >= data_at) left = uint64_t(end - data_at);
        fseek(f, data_at, SEEK_SET);
    }
    const uint64_t need = uint64_t(w) * uint64_t(h) * uint64_t(ch); // < 2^64: w, h < 2^31, ch <= 3
    if (need > left) {
        fclose(f);
        return RT_ERR_IO;
    }
    size_t n = size_t(w) * size_t(h) * 3;
    std::vector<uint8_t> bytes;
    try {
        bytes.resize(size_t(need));
    } catch (const std::exception&) {
        fclose(f);
        return RT_ERR_OOM;
    }
    ok = fread(bytes.data(), 1, bytes.size(), f) == bytes.size();
    fclose(f);
    if (!ok) return RT_ERR_IO;
    float* rgb = static_cast<float*>(malloc(n * sizeof(float)));
    if (!rgb) return RT_ERR_OOM;
    if (ch == 3) {
        for (size_t i = 0; i < n; ++i) rgb[i] = float(bytes[i]) / 255.0f;
    } else { // grey -> RGB: what rt_image_to_rgb does with a 1-channel stbi_loadf result
        for (size_t i = 0; i < bytes.size(); ++i) rgb[3 * i] = rgb[3 * i + 1] = rgb[3 * i + 2] = float(bytes[i]) / 255.0f;
    }
    *out_rgb = rgb;
    *width = w;
    *height = h;
    return RT_OK;
}

// What stbi_loadf hands back for a file with `channels` components, as the 3-component image image_texture indexes
// (texture.h:118-132 assumes RGB, main.cu:384 allocates w*h*ch): grey -> (g,g,g), grey+alpha -> (g,g,g), RGB -> copy,
// RGBA -> alpha dropped (stb_image.h stbi__convert_format semantics for req_comp = 3).
rt_status rt_image_to_rgb(const float* data, int32_t width, int32_t height, int32_t channels, float* out_rgb) {
    if (!data || !out_rgb || width <= 0 || height <= 0 || channels < 1 || channels > 4) return RT_ERR_INVALID_ARG;
    const size_t n = size_t(width) * size_t(height);
    for (size_t i = 0; i < n; ++i) {
        const float* p = data + i * size_t(channels);
        float* o = out_rgb + i * 3;
        if (channels <= 2) {
            o[0] = o[1] = o[2] = p[0];
        } else {
            o[0] = p[0];
            o[1] = p[1];
            o[2] = p[2];
        }
    }
    return RT_OK;
}

void rt_free(void* p) { free(p); }

rt_status rt_builtin_scene(const char* name, const float* image_rgb, int32_t image_w, int32_t image_h, uint32_t n,
                           uint32_t bvh_mode, rt_scene_desc** out) {
    if (!name || !out) return RT_ERR_INVALID_ARG;
    *out = nullptr;
    try {
        rt::arena A;
        rt::scenes::built b;
        std::string nm(name);
        if (nm == "earth_emitter") {
            if (!image_rgb || image_w <= 0 || image_h <= 0) return RT_ERR_INVALID_ARG;
            b = rt::scenes::earth_emitter(A, image_rgb, image_w, image_h, bvh_mode);
        } else if (nm == "hdr_sphere") {
            if (!image_rgb || image_w <= 0 || image_h <= 0) return RT_ERR_INVALID_ARG;
            b = rt::scenes::hdr_sphere(A, image_rgb, image_w, image_h);
        } else if (nm == "book1_final") {
            b = rt::scenes::book1_final(A, bvh_mode);
        } else if (nm == "perlin_motion") {
            b = rt::scenes::perlin_motion(A, bvh_mode);
        } else if (nm == "random_spheres") {
            b = rt::scenes::random_spheres(A, n, bvh_mode);
        } else {
            return RT_ERR_INVALID_ARG;
        }
        OwnedDesc* od = new OwnedDesc();
        od->fs = rt::flatten(*b.list, *b.cam);
        for (const rt_image& im : od->fs.images)
            od->image_data.emplace_back(im.rgb, im.rgb + size_t(im.width) * size_t(im.height) * 3);
        od->bind();
        *out = &od->desc;
        return RT_OK;
    } catch (const std::bad_alloc&) {
        return RT_ERR_OOM;
    } catch (const std::exception&) {
        return RT_ERR_INVALID_ARG;
    }
}

// Runtime scene front-end (SURVEY.md 8f-3): JSON text -> façade objects -> flattened description.
rt_status rt_scene_desc_from_json(rt_context* ctx, const char* json_text, const char* base_dir, rt_render_params* render,
                                  rt_scene_desc** out) {
    if (!json_text || !out) return RT_ERR_INVALID_ARG;
    *out = nullptr;
    OwnedDesc* od = nullptr;
    try {
        rt::arena A;
        rt::scenes::json_scene js;
        auto load = [ctx](const std::string& path, std::vector<float>& rgb, int& w, int& h) {
            float* p = nullptr;
            int32_t ww = 0, hh = 0;
            if (rt_image_load(ctx, path.c_str(), &p, &ww, &hh) != RT_OK) return false; // PPM/PGM, or JPEG when ctx != NULL
            rgb.assign(p, p + size_t(ww) * size_t(hh) * 3);
            free(p);
            w = ww;
            h = hh;
            return true;
        };
        rt::scenes::scene_from_json(json_text, base_dir ? base_dir : "", load, A, js, render);
        od = new OwnedDesc();
        od->fs = rt::flatten(*js.b.list, *js.b.cam);
        for (const rt_image& im : od->fs.images)
            od->image_data.emplace_back(im.rgb, im.rgb + size_t(im.width) * size_t(im.height) * 3);
        od->bind();
        *out = &od->desc;
        return RT_OK;
    } catch (const std::bad_alloc&) {
        delete od;
        return RT_ERR_OOM;
    } catch (const std::exception& e) {
        delete od;
        rtd::set_error_message(e.what());
        return RT_ERR_INVALID_ARG;
    }
}

rt_status rt_scene_desc_from_json_file(rt_context* ctx, const char* path, rt_render_params* render, rt_scene_desc** out) {
    if (!path || !out) return RT_ERR_INVALID_ARG;
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) {
        rtd::set_error_message((std::string("cannot open ") + path).c_str());
        return RT_ERR_IO;
    }
    std::string text;
    char buf[65536];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) text.append(buf, n);
    fclose(f);
    std::string dir(path);
    const size_t slash = dir.find_last_of('/');
    dir = slash == std::string::npos ? std::string() : dir.substr(0, slash);
    return rt_scene_desc_from_json(ctx, text.c_str(), dir.c_str(), render, out);
}

void rt_scene_desc_free(rt_scene_desc* desc) {
    if (desc) delete reinterpret_cast<OwnedDesc*>(desc);
}

// ---- flat scene file: shared with oracle/ref_harness.cu ----
//   u32 'RTSC', u32 version(1), u32 n_spheres, n_materials, n_textures, n_images, bvh_mode,
//   rt_camera, spheres[], materials[], textures[], then per image: i32 w, i32 h, float rgb[w*h*3]
rt_status rt_scene_desc_save(const rt_scene_desc* d, const char* path) {
    if (!d || !path) return RT_ERR_INVALID_ARG;
    FILE* f = fopen(path, "wb");
    if (!f) return RT_ERR_IO;
    uint32_t hdr[7] = {0x43535452u, 1u, d->n_spheres, d->n_materials, d->n_textures, d->n_images, d->bvh_mode};
    bool ok = fwrite(hdr, sizeof hdr, 1, f) == 1;
    ok = ok && fwrite(&d->camera, sizeof(rt_camera), 1, f) == 1;
    ok = ok && (d->n_spheres == 0 || fwrite(d->spheres, sizeof(rt_sphere), d->n_spheres, f) == d->n_spheres);
    ok = ok && (d->n_materials == 0 || fwrite(d->materials, sizeof(rt_material), d->n_materials, f) == d->n_materials);
    ok = ok && (d->n_textures == 0 || fwrite(d->textures, sizeof(rt_texture), d->n_textures, f) == d->n_textures);
    for (uint32_t i = 0; ok && i < d->n_images; ++i) {
        int32_t wh[2] = {d->images[i].width, d->images[i].height};
        size_t n = size_t(wh[0]) * size_t(wh[1]) * 3;
        ok = fwrite(wh, sizeof wh, 1, f) == 1 && fwrite(d->images[i].rgb, sizeof(float), n, f) == n;
    }
    ok = (fclose(f) == 0) && ok;
    return ok ? RT_OK : RT_ERR_IO;
}

rt_status rt_scene_desc_load(const char* path, rt_scene_desc** out) {
    if (!path || !out) return RT_ERR_INVALID_ARG;
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return RT_ERR_IO;
    OwnedDesc* od = nullptr;
    try {
        od = new OwnedDesc();
        // the counts of a damaged file must not size an allocation: everything is checked against the bytes that are there
        uint64_t left = 0;
        if (fseek(f, 0, SEEK_END) == 0) {
            const long end = ftell(f);
            left = end > 0 ? uint64_t(end) : 0;
        }
        rewind(f);
        uint32_t hdr[7];
        bool ok = left >= sizeof hdr + sizeof(rt_camera) && fread(hdr, sizeof hdr, 1, f) == 1 && hdr[0] == 0x43535452u && hdr[1] == 1u;
        ok = ok && fread(&od->fs.cam, sizeof(rt_camera), 1, f) == 1;
        if (ok) {
            left -= sizeof hdr + sizeof(rt_camera);
            const uint64_t arrays = uint64_t(hdr[2]) * sizeof(rt_sphere) + uint64_t(hdr[3]) * sizeof(rt_material) +
                                    uint64_t(hdr[4]) * sizeof(rt_texture);
            ok = arrays <= left && uint64_t(hdr[5]) * (2 * sizeof(int32_t)) <= left - arrays;
            if (ok) left -= arrays;
        }
        if (ok) {
            od->fs.spheres.resize(hdr[2]);
            od->fs.materials.resize(hdr[3]);
            od->fs.textures.resize(hdr[4]);
            od->fs.images.resize(hdr[5]);
            od->fs.bvh_mode = hdr[6];
            ok = (hdr[2] == 0 || fread(od->fs.spheres.data(), sizeof(rt_sphere), hdr[2], f) == hdr[2]) &&
                 (hdr[3] == 0 || fread(od->fs.materials.data(), sizeof(rt_material), hdr[3], f) == hdr[3]) &&
                 (hdr[4] == 0 || fread(od->fs.textures.data(), sizeof(rt_texture), hdr[4], f) == hdr[4]);
        }
        for (uint32_t i = 0; ok && i < hdr[5]; ++i) {
            int32_t wh[2];
            ok = left >= sizeof wh && fread(wh, sizeof wh, 1, f) == 1 && wh[0] > 0 && wh[1] > 0;
            if (!ok) break;
            left -= sizeof wh;
            const uint64_t n = uint64_t(wh[0]) * uint64_t(wh[1]) * 3; // < 2^64: both factors are below 2^31
            ok = n <= left / sizeof(float);
            if (!ok) break;
            left -= n * sizeof(float);
            od->image_data.emplace_back(n);
            ok = fread(od->image_data.back().data(), sizeof(float), n, f) == n;
            od->fs.images[i] = rt_image{nullptr, wh[0], wh[1]};
        }
        fclose(f);
        f = nullptr;
        if (!ok) {
            delete od;
            return RT_ERR_IO;
        }
        od->bind();
        *out = &od->desc;
        return RT_OK;
    } catch (const std::bad_alloc&) {
        if (f) fclose(f);
        delete od;
        return RT_ERR_OOM;
    } catch (const std::exception& e) { // nothing may propagate through the C ABI
        if (f) fclose(f);
        delete od;
        rtd::set_error_message(e.what());
        return RT_ERR_IO;
    }
}

} // extern "C"
