// ORACLE — TEST INFRASTRUCTURE ONLY.  C entry points (ctypes) over oracle.cpp.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstring>
#include <thread>
#include <vector>

#include "oracle.hpp"

using namespace orc;

static inline V3 fr(rt_vec3 a) { return V3{a.x, a.y, a.z}; }
static inline rt_vec3 to(V3 a) { return rt_vec3{a.x, a.y, a.z}; }

static void mat_out(const Mat4& m, double* out16) {
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) out16[i * 4 + j] = m.m[i][j];
}
static Mat4 mat_in(const double* in16) {
    Mat4 m;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) m.m[i][j] = in16[i * 4 + j];
    return m;
}

extern "C" {

// ---- algebra ---------------------------------------------------------------------------------
void orc_mat_mul(const double* a16, const double* b16, double* out16) {
    mat_out(mat_mul(mat_in(a16), mat_in(b16)), out16);
}
void orc_mat_rotate(rt_vec3 deg, double* out16) { mat_out(mat_rotate(fr(deg)), out16); }
void orc_transform_new(rt_vec3 translate, rt_vec3 rotate, rt_vec3 scale, double* direct16, double* inverse16) {
    Mat4 d, i;
    inversable_transform_new(fr(translate), fr(rotate), fr(scale), &d, &i);
    mat_out(d, direct16);
    mat_out(i, inverse16);
}
rt_vec3 orc_transform_point(const double* m16, rt_vec3 p) { return to(transform_point(mat_in(m16), fr(p))); }
rt_vec3 orc_transform_vector(const double* m16, rt_vec3 p) { return to(transform_vector(mat_in(m16), fr(p))); }
rt_vec3 orc_transform_normal(const double* m16, rt_vec3 p) { return to(transform_normal(mat_in(m16), fr(p))); }
void orc_aabb_transform(rt_vec3 mn, rt_vec3 mx, const double* m16, rt_vec3* omn, rt_vec3* omx) {
    V3 a, b;
    aabb_transform(fr(mn), fr(mx), mat_in(m16), &a, &b);
    *omn = to(a);
    *omx = to(b);
}
rt_vec3 orc_reflect(rt_vec3 v, rt_vec3 n) { return to(reflect(fr(v), fr(n))); }
rt_vec3 orc_refract(rt_vec3 v, rt_vec3 n, double ratio) { return to(refract(fr(v), fr(n), ratio)); }

// ---- camera ----------------------------------------------------------------------------------
void orc_camera_new(rt_vec3 position, rt_vec3 direction, rt_vec3 up, double focal_length, double fov_rad,
                    rt_camera* out) {
    *out = camera_new(fr(position), fr(direction), fr(up), focal_length, fov_rad);
}
double orc_raycaster_pixel_resolution(const rt_camera* cam, rt_image_params img) {
    return raycaster_new(*cam, img).pixel_resolution;
}
void orc_raycaster_get_ray(const rt_camera* cam, rt_image_params img, double x, double y, rt_ray* out) {
    Ray r = raycaster_get_ray(raycaster_new(*cam, img), x, y);
    out->origin = to(r.origin);
    out->direction = to(r.direction);
}

// ---- rng -------------------------------------------------------------------------------------
void orc_philox4x32_10(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4) {
    philox4x32_10(ctr4, key2, out4);
}
// the first n doubles of the shared stream (seed; pixel, sample, event)
void orc_philox_stream(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t event, uint32_t n, double* out) {
    PathRng r;
    r.mode = RNG_PHILOX;
    r.key[0] = (uint32_t)seed;
    r.key[1] = (uint32_t)(seed >> 32);
    r.pixel = pixel;
    r.sample = sample;
    r.begin_event(event);
    for (uint32_t i = 0; i < n; i++) out[i] = r.next();
}

// ---- surfaces --------------------------------------------------------------------------------
double orc_surface_func(const double* params8, rt_vec3 p) { return surface_func(params8, fr(p)); }
rt_vec3 orc_surface_gradient(const double* params8, rt_vec3 p) { return to(surface_gradient(params8, fr(p))); }

// ---- scene handle ----------------------------------------------------------------------------
void* orc_scene_create(const rt_scene_desc* d) {
    Scene* s = new Scene();
    if (!scene_from_desc(d, s)) {
        delete s;
        return nullptr;
    }
    return s;
}
void orc_scene_destroy(void* s) { delete (Scene*)s; }
void orc_scene_build_bvh(void* s, uint64_t seed) { build_bvh(*(Scene*)s, seed); }
void orc_shape_bounding_box(void* s, uint32_t i, rt_vec3* mn, rt_vec3* mx) {
    V3 a, b;
    shape_bounding_box(((Scene*)s)->shapes[i], &a, &b);
    *mn = to(a);
    *mx = to(b);
}

// Batched nearest hit with the ShapeCollection semantics (use_bvh = 0) or the BvhNode semantics
// (use_bvh = 1; orc_scene_build_bvh first).  counters_out: segments, shape_tests, march_steps,
// march_rays, aabb_tests.  Returns wall seconds.
double orc_intersect_batch(void* sv, const rt_ray* rays, uint64_t n, double t_min, double t_max, int use_bvh,
                           uint32_t threads, int32_t* shape_index, double* t, rt_vec3* normal, rt_vec3* point,
                           double* uv, uint8_t* front_face, uint64_t* counters_out) {
    const Scene& sc = *(Scene*)sv;
    if (threads == 0) threads = 1;
    std::vector<Counters> cs(threads);
    auto t0 = std::chrono::steady_clock::now();
    auto work = [&](uint32_t tid) {
        uint64_t lo = n * tid / threads, hi = n * (tid + 1) / threads;
        Counters* c = counters_out ? &cs[tid] : nullptr;
        for (uint64_t i = lo; i < hi; i++) {
            Ray r{fr(rays[i].origin), fr(rays[i].direction)};
            Hit h;
            if (c) c->segments++;
            bool ok = use_bvh ? bvh_ray_hit(sc, r, t_min, t_max, &h, c)
                              : collection_ray_intersect(sc, r, t_min, t_max, &h, c);
            if (shape_index) shape_index[i] = ok ? h.shape : -1;
            if (!ok) {
                if (t) t[i] = 0.0;
                if (normal) normal[i] = rt_vec3{0, 0, 0};
                if (point) point[i] = rt_vec3{0, 0, 0};
                if (uv) uv[2 * i] = uv[2 * i + 1] = 0.0;
                if (front_face) front_face[i] = 0;
                continue;
            }
            if (t) t[i] = h.distance;
            if (normal) normal[i] = to(h.normal);
            if (point) point[i] = to(h.point);
            if (uv) { uv[2 * i] = h.u; uv[2 * i + 1] = h.v; }
            if (front_face) front_face[i] = h.is_front_face ? 1 : 0;
        }
    };
    std::vector<std::thread> th;
    for (uint32_t k = 1; k < threads; k++) th.emplace_back(work, k);
    work(0);
    for (auto& x : th) x.join();
    auto t1 = std::chrono::steady_clock::now();
    if (counters_out) {
        Counters tot;
        for (auto& c : cs) tot.add(c);
        counters_out[0] = tot.segments;
        counters_out[1] = tot.shape_tests;
        counters_out[2] = tot.march_steps;
        counters_out[3] = tot.march_rays;
        counters_out[4] = tot.aabb_tests;
    }
    return std::chrono::duration<double>(t1 - t0).count();
}

// Threaded frame render (the CPU baseline).  rng_mode 0 = shared Philox schedule, 1 = independent.
double orc_render(void* sv, const rt_camera* cam, uint32_t width, uint32_t height, uint32_t spp, uint32_t depth,
                  uint64_t seed, int rng_mode, int use_bvh, uint32_t threads, uint32_t stride_x,
                  uint32_t stride_y, rt_vec3* buffer, uint64_t* counters_out) {
    RenderOptions o;
    o.image = rt_image_params{width, height};
    o.samples_number = spp;
    o.max_depth = depth;
    o.seed = seed;
    o.rng = rng_mode ? RNG_XOSHIRO : RNG_PHILOX;
    o.use_bvh = use_bvh != 0;
    o.threads = threads;
    o.stride_x = stride_x;
    o.stride_y = stride_y;
    Counters c;
    double s = render(*(Scene*)sv, *cam, o, buffer, counters_out ? &c : nullptr);
    if (counters_out) {
        counters_out[0] = c.segments;
        counters_out[1] = c.shape_tests;
        counters_out[2] = c.march_steps;
        counters_out[3] = c.march_rays;
        counters_out[4] = c.aabb_tests;
    }
    return s;
}

// renderer::trace_pixel_samples (renderer/mod.rs:151-155) on caller-supplied rays, Philox schedule
void orc_trace_pixel_samples(void* sv, const rt_ray* rays, uint32_t n_rays, uint32_t depth, uint64_t seed,
                             uint32_t pixel_index, int use_bvh, rt_vec3* mean_out) {
    const Scene& sc = *(Scene*)sv;
    PathRng rng;
    rng.mode = RNG_PHILOX;
    rng.key[0] = (uint32_t)seed;
    rng.key[1] = (uint32_t)(seed >> 32);
    rng.pixel = pixel_index;
    V3 acc = v3(0, 0, 0);
    for (uint32_t s = 0; s < n_rays; s++) {
        rng.sample = s;
        Ray r{fr(rays[s].origin), fr(rays[s].direction)};
        V3 col = ray_color(sc, use_bvh != 0, r, depth, rng, 0, nullptr);
        acc.x += col.x; acc.y += col.y; acc.z += col.z;
    }
    *mean_out = to(acc / (double)n_rays);
}

// Per-sample radiance of a list of pixels with the Philox schedule (raygen included), samples sample_base ..
// sample_base + n_samples - 1 of each: lets a test compare individual GPU paths with the oracle.
// colors_out[i * n_samples + s] = sample sample_base + s of pixel pixel_index[i] (= x + y * width).  Pixels are
// spread over `threads` worker threads; every path is computed exactly as orc_render computes it.
void orc_pixels_sample_colors(void* sv, const rt_camera* cam, uint32_t width, uint32_t height, uint64_t n_pixels,
                              const uint32_t* pixel_index, uint32_t sample_base, uint32_t n_samples, uint32_t depth,
                              uint64_t seed, uint32_t threads, rt_vec3* colors_out) {
    const Scene& sc = *(Scene*)sv;
    const RayCaster rc = raycaster_new(*cam, rt_image_params{width, height});
    std::atomic<uint64_t> next{0};
    auto work = [&]() {
        PathRng rng;
        rng.mode = RNG_PHILOX;
        rng.key[0] = (uint32_t)seed;
        rng.key[1] = (uint32_t)(seed >> 32);
        for (uint64_t i = next++; i < n_pixels; i = next++) {
            const uint32_t p = pixel_index[i], x = p % width, y = p / width;
            rng.pixel = p;
            for (uint32_t s = 0; s < n_samples; s++) {
                rng.sample = sample_base + s;
                rng.begin_event(0);
                double u = rng.next(), v = rng.next();
                Ray r = raycaster_get_ray(rc, (double)x + u, (double)y + v);
                colors_out[i * n_samples + s] = to(ray_color(sc, false, r, depth, rng, 0, nullptr));
            }
        }
    };
    if (threads == 0) threads = 1;
    if (threads > n_pixels) threads = (uint32_t)std::max<uint64_t>(n_pixels, 1);
    std::vector<std::thread> th;
    for (uint32_t k = 1; k < threads; k++) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}

// Per-ray radiance of caller-supplied rays in groups (trace_pixel_samples_group): group g is rays offsets[g] ..
// offsets[g + 1] - 1, and ray r of it is traced with the RNG key (seed; pixel_index[g], r - offsets[g]), as
// orc_trace_pixel_samples keys its rays.  The rays are used as given (not normalised).  Groups are spread over
// `threads` worker threads; colors_out[r] = the FP64 colour of ray r.
void orc_groups_sample_colors(void* sv, const rt_ray* rays, uint64_t n_rays, const uint64_t* offsets,
                              const uint32_t* pixel_index, uint64_t n_groups, uint32_t depth, uint64_t seed,
                              uint32_t threads, rt_vec3* colors_out) {
    (void)n_rays;
    const Scene& sc = *(Scene*)sv;
    std::atomic<uint64_t> next{0};
    auto work = [&]() {
        PathRng rng;
        rng.mode = RNG_PHILOX;
        rng.key[0] = (uint32_t)seed;
        rng.key[1] = (uint32_t)(seed >> 32);
        for (uint64_t g = next++; g < n_groups; g = next++) {
            rng.pixel = pixel_index[g];
            for (uint64_t r = offsets[g]; r < offsets[g + 1]; r++) {
                rng.sample = (uint32_t)(r - offsets[g]);
                Ray ray{fr(rays[r].origin), fr(rays[r].direction)};
                colors_out[r] = to(ray_color(sc, false, ray, depth, rng, 0, nullptr));
            }
        }
    };
    if (threads == 0) threads = 1;
    if (threads > n_groups) threads = (uint32_t)std::max<uint64_t>(n_groups, 1);
    std::vector<std::thread> th;
    for (uint32_t k = 1; k < threads; k++) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}

// The same for one pixel (x, y), samples 0 .. spp - 1, on the calling thread.
void orc_pixel_sample_colors(void* sv, const rt_camera* cam, uint32_t width, uint32_t height, uint32_t x,
                             uint32_t y, uint32_t spp, uint32_t depth, uint64_t seed, rt_vec3* colors_out) {
    const uint32_t p = x + y * width;
    orc_pixels_sample_colors(sv, cam, width, height, 1, &p, 0, spp, depth, seed, 1, colors_out);
}

uint32_t orc_hardware_threads(void) {
    unsigned n = std::thread::hardware_concurrency();
    return n ? n : 1;
}

// ---- per-shape hits of one ray: Shape::ray_hit for EVERY shape with max_t = +inf (no shrinking), so that
// tests can check the GPU core's conservative culling pair by pair.  hits[i] = 1 when shape i returns Some.
// A ray-marched shape counts as hit as soon as its bound is entered (intersect_bound returns Some): that is
// the decision the pre-test in front of it must never contradict.
void orc_shape_hits(const Scene* sc, const rt_ray* ray, double min_t, uint8_t* hits) {
    Ray r;
    r.origin = fr(ray->origin);
    r.direction = fr(ray->direction);
    for (size_t i = 0; i < sc->shapes.size(); i++) {
        const Shape& s = sc->shapes[i];
        if (s.kind == RT_SHAPE_MARCH) {
            Ray local;
            local.origin = transform_point(s.inverse, r.origin);
            local.direction = transform_vector(s.inverse, r.direction);
            double start, end;
            hits[i] = march_intersect_bound(s, local, &start, &end) ? 1 : 0;
        } else {
            Hit h;
            hits[i] = shape_ray_hit(s, (int)i, r, min_t, INFINITY, &h, nullptr) ? 1 : 0;
        }
    }
}

void orc_solve_quartic(double a, double b, double c, double d, double e, double* re4, double* im4) {
    solve_quantic_equation(a, b, c, d, e, re4, im4);
}

// ---- Perlin noise (src/algebra/noise.rs) ---------------------------------------------------------
double orc_perlin_noise(const rt_perlin* pn, rt_vec3 p) { return perlin_noise(*pn, fr(p)); }
double orc_perlin_turb(const rt_perlin* pn, rt_vec3 p, int depth) { return perlin_turb(*pn, fr(p), depth); }

}  // extern "C"
