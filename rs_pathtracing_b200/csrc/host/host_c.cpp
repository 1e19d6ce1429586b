// C shim (include/rt_b200_host.h) over the C++ host mirror, for ctypes and C embedders.
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>

#include <algorithm>
#include <cstdio>
#include <vector>
#include "../../../include/rt_b200_host.h"
#include "ray_tracing.hpp"

using namespace ray_tracing;

struct rth_scene {
    std::shared_ptr<world::Scene> scene;
};
struct rth_renderer {
    std::unique_ptr<renderer::GpuRenderer> r;
};

static thread_local std::string g_err;

template <class F>
static int guarded(F&& f) {
    try {
        f();
        return RT_OK;
    } catch (const std::exception& e) {
        g_err = e.what();
        return RT_ERR_INVALID;
    } catch (...) {
        g_err = "unknown error";
        return RT_ERR_INVALID;
    }
}

static algebra::Vector3d V(rt_vec3 a) { return algebra::Vector3d(a.x, a.y, a.z); }

extern "C" {

const char* rth_last_error(void) { return g_err.c_str(); }

void rth_set_image_loader(rth_image_loader fn) {
    // same signature modulo the bool/int return type
    world::set_image_loader(reinterpret_cast<world::ImageLoaderFn>(fn));
}

int rth_scene_from_json(const char* json_text, uint64_t seed, int add_random_spheres, rth_scene** out) {
    if (!json_text || !out) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] {
        auto sc = world::Scene::from_json(json_text, seed, add_random_spheres != 0);
        *out = new rth_scene{sc};
    });
}
void rth_scene_free(rth_scene* s) { delete s; }
int rth_scene_desc(rth_scene* s, rt_scene_desc* out) {
    if (!s || !out) { g_err = "null argument"; return RT_ERR_INVALID; }
    *out = s->scene->flat().desc();
    return RT_OK;
}
int rth_scene_camera(rth_scene* s, rt_camera* out) {
    if (!s || !out) { g_err = "null argument"; return RT_ERR_INVALID; }
    *out = s->scene->camera().to_pod();
    return RT_OK;
}
uint32_t rth_scene_shape_count(rth_scene* s) { return s ? s->scene->shape_count() : 0; }
const char* rth_scene_shape_name(rth_scene* s, uint32_t i) {
    if (!s || i >= s->scene->flat().shape_names.size()) return "";
    return s->scene->flat().shape_names[i].c_str();
}
const char* rth_scene_material_name(rth_scene* s, uint32_t i) {
    if (!s || i >= s->scene->flat().material_names.size()) return "";
    return s->scene->flat().material_names[i].c_str();
}
int rth_scene_assign_material(rth_scene* s, uint32_t shape_index, const char* name) {
    if (!s || !name) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { s->scene->assign_material(shape_index, name); });
}
int rth_scene_set_transforms(rth_scene* s, uint32_t n, const uint32_t* index, const double* direct16,
                             const double* inverse16) {
    if (!s) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { s->scene->set_transforms(n, index, direct16, inverse16); });
}
int rth_scene_device(rth_scene* s, int device, rt_scene** out) {
    if (!s || !out) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { *out = s->scene->device_scene(device); });
}

int rth_scene_device_multi(rth_scene* s, int n_devices, const int* device_ids, rt_scene** out) {
    if (!s || !out || !device_ids || n_devices < 1) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { *out = s->scene->device_scene(std::vector<int>(device_ids, device_ids + n_devices)); });
}

int rth_camera_new(rt_vec3 position, rt_vec3 direction, rt_vec3 up, double focal_length, double fov_rad,
                   rt_camera* out) {
    if (!out) { g_err = "null argument"; return RT_ERR_INVALID; }
    *out = camera::Camera(V(position), V(direction), V(up), focal_length, fov_rad).to_pod();
    return RT_OK;
}
int rth_transform_new(rt_vec3 translate, rt_vec3 rotate_deg, rt_vec3 scale, double* direct16, double* inverse16) {
    algebra::transform::InversableTransform t(V(translate), V(rotate_deg), V(scale));
    if (direct16) memcpy(direct16, t.direct.m, sizeof(double) * 16);
    if (inverse16) memcpy(inverse16, t.inverse.m, sizeof(double) * 16);
    return RT_OK;
}

int rth_renderer_new(rth_scene* s, uint32_t thread_number, uint32_t depth, int device, uint64_t seed,
                     rth_renderer** out) {
    if (!s || !out) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] {
        auto r = std::make_unique<renderer::GpuRenderer>(s->scene, thread_number, depth, device, seed);
        *out = new rth_renderer{std::move(r)};
    });
}
int rth_renderer_new_multi(rth_scene* s, uint32_t thread_number, uint32_t depth, int n_devices, const int* device_ids,
                           uint64_t seed, rth_renderer** out) {
    if (!s || !out || !device_ids || n_devices < 1) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] {
        auto r = std::make_unique<renderer::GpuRenderer>(s->scene, thread_number, depth,
                                                         std::vector<int>(device_ids, device_ids + n_devices), seed);
        *out = new rth_renderer{std::move(r)};
    });
}
void rth_renderer_free(rth_renderer* r) { delete r; }
int rth_renderer_start_rendering(rth_renderer* r, const rt_camera* cam, rt_image_params img, uint32_t spp) {
    if (!r || !cam) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] {
        auto c = std::make_shared<camera::Camera>(camera::Camera::from_pod(*cam));
        r->r->start_rendering(c, camera::ImageParams{img.width, img.height}, spp);
    });
}
int rth_renderer_render_step(rth_renderer* r, rt_vec3* buffer, uint64_t len, int* done) {
    if (!r || !buffer || !done) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { *done = r->r->render_step((algebra::Vector3d*)buffer, (size_t)len) ? 1 : 0; });
}
int rth_renderer_stop_rendering(rth_renderer* r) {
    if (!r) { g_err = "null argument"; return RT_ERR_INVALID; }
    return guarded([&] { r->r->stop_rendering(); });
}

// ---- PNG output ------------------------------------------------------------------------------
static uint32_t crc32_update(uint32_t crc, const uint8_t* p, size_t n) {
    static uint32_t table[256];
    static bool init = false;
    if (!init) {
        for (uint32_t i = 0; i < 256; i++) {
            uint32_t c = i;
            for (int k = 0; k < 8; k++) c = (c & 1) ? 0xEDB88320u ^ (c >> 1) : c >> 1;
            table[i] = c;
        }
        init = true;
    }
    for (size_t i = 0; i < n; i++) crc = table[(crc ^ p[i]) & 0xff] ^ (crc >> 8);
    return crc;
}
static void put_be32(std::vector<uint8_t>& v, uint32_t x) {
    v.push_back((uint8_t)(x >> 24)); v.push_back((uint8_t)(x >> 16)); v.push_back((uint8_t)(x >> 8)); v.push_back((uint8_t)x);
}
static void png_chunk(std::vector<uint8_t>& out, const char* type, const std::vector<uint8_t>& data) {
    put_be32(out, (uint32_t)data.size());
    size_t at = out.size();
    out.insert(out.end(), type, type + 4);
    out.insert(out.end(), data.begin(), data.end());
    put_be32(out, crc32_update(0xFFFFFFFFu, out.data() + at, out.size() - at) ^ 0xFFFFFFFFu);
}

int rth_save_png(const char* path, const uint8_t* rgba, uint32_t width, uint32_t height) {
    if (!path || !rgba || width == 0 || height == 0) { g_err = "null or empty argument"; return RT_ERR_INVALID; }
    return guarded([&] {
        // raw scanlines: filter byte 0 + width * 4 bytes
        std::vector<uint8_t> raw;
        raw.reserve((size_t)height * ((size_t)width * 4 + 1));
        for (uint32_t y = 0; y < height; y++) {
            raw.push_back(0);
            raw.insert(raw.end(), rgba + (size_t)y * width * 4, rgba + (size_t)(y + 1) * width * 4);
        }
        // zlib stream of stored (uncompressed) deflate blocks
        std::vector<uint8_t> z = {0x78, 0x01};
        uint32_t a = 1, b = 0;  // Adler-32
        for (size_t i = 0; i < raw.size(); i++) { a = (a + raw[i]) % 65521u; b = (b + a) % 65521u; }
        for (size_t off = 0; off < raw.size(); off += 65535) {
            size_t n = std::min<size_t>(65535, raw.size() - off);
            z.push_back(off + n >= raw.size() ? 1 : 0);
            z.push_back((uint8_t)(n & 0xff)); z.push_back((uint8_t)(n >> 8));
            z.push_back((uint8_t)(~n & 0xff)); z.push_back((uint8_t)((~n >> 8) & 0xff));
            z.insert(z.end(), raw.begin() + off, raw.begin() + off + n);
        }
        put_be32(z, (b << 16) | a);
        std::vector<uint8_t> out = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
        std::vector<uint8_t> ihdr;
        put_be32(ihdr, width);
        put_be32(ihdr, height);
        ihdr.insert(ihdr.end(), {8, 6, 0, 0, 0});  // 8 bit, RGBA, deflate, no filter, no interlace
        png_chunk(out, "IHDR", ihdr);
        png_chunk(out, "IDAT", z);
        png_chunk(out, "IEND", {});
        FILE* f = fopen(path, "wb");
        if (!f) throw std::runtime_error(std::string("cannot open ") + path);
        size_t w = fwrite(out.data(), 1, out.size(), f);
        fclose(f);
        if (w != out.size()) throw std::runtime_error(std::string("short write to ") + path);
    });
}

}  // extern "C"
