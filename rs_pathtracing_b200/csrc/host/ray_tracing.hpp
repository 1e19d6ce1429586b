// Host-side mirror of the reference crate's public interface for the hot path, in C++ because
// the image has no Rust toolchain (the reference is compiled code -> the host side is C++).
// Names, argument meaning and error behaviour follow the crate `ray_tracing`:
//   algebra::Vector3d / transform::{Transform, InversableTransform}   src/algebra/{mod,transform}.rs
//   camera::{Camera, ray_caster::ImageParams}                         src/camera/{mod,ray_caster}.rs
//   world::{Scene, ray::Ray}                                          src/world/{mod,ray,json_models}.rs
//   renderer::{Renderer, GpuRenderer}                                 src/renderer/{mod,step_by_step}.rs
// Everything below the Renderer / Scene::closest_hit seam runs on the GPU through the C ABI in
// include/rt_b200.h; nothing in this layer computes an intersection or a colour on the CPU.
#pragma once
#include <cstdint>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../../include/rt_b200.h"

namespace ray_tracing {

namespace algebra {

// src/algebra/mod.rs:23-28 — layout-identical to rt_vec3
struct Vector3d {
    double x, y, z;
    Vector3d() : x(0), y(0), z(0) {}
    Vector3d(double x_, double y_, double z_) : x(x_), y(y_), z(z_) {}
    Vector3d cross(const Vector3d& o) const;   // :99-105
    Vector3d normalize() const;                // :107-110
    double squared_length() const;             // :112-115
    double length() const;                     // :117-120
};

namespace transform {

// src/algebra/transform.rs:189-190
struct Transform {
    double m[4][4];
    static Transform unit();
    static Transform translate(const Vector3d& v);      // :316-323
    static Transform scale(const Vector3d& v);          // :325-332
    static Transform rotate(const Vector3d& degrees);   // :334-358  roll(x)*pitch(y)*yaw(z)
    static Transform rotate_inverse(const Vector3d& degrees);  // :360-362
    static Transform rotate_roll(double degrees);       // :364-372
    static Transform rotate_pitch(double degrees);      // :374-382
    static Transform rotate_yaw(double degrees);        // :384-392
    Transform operator*(const Transform& rhs) const;    // :553-570
    Vector3d transform_point(const Vector3d& p) const;  // :394-409
    Vector3d transform_vector(const Vector3d& v) const; // :411-417
    Vector3d transform_normal(const Vector3d& n) const; // :419-425
};

// src/algebra/transform.rs:6-23
struct InversableTransform {
    Vector3d translate, rotate, scale;
    Transform direct, inverse;
    InversableTransform() : direct(Transform::unit()), inverse(Transform::unit()) {}
    InversableTransform(const Vector3d& translate, const Vector3d& rotate, const Vector3d& scale);
};

}  // namespace transform
}  // namespace algebra

namespace camera {

// src/camera/ray_caster.rs:10-14
struct ImageParams {
    uint32_t width, height;
};

// src/camera/mod.rs:36-46
class Camera {
public:
    Camera() : fov_(0), focal_length_(0) {}
    // Camera::new, :71-88 (fov in radians)
    Camera(const algebra::Vector3d& position, const algebra::Vector3d& direction,
           const algebra::Vector3d& up_vector, double focal_length, double fov);
    const algebra::Vector3d& position() const { return position_; }
    const algebra::Vector3d& direction() const { return direction_; }
    const algebra::Vector3d& up() const { return up_; }
    const algebra::Vector3d& rigth() const { return rigth_; }   // sic, :45
    double fov() const { return fov_; }
    double focal_length() const { return focal_length_; }
    void set_position(const algebra::Vector3d& p) { position_ = p; }   // :129-131
    void set_direction(const algebra::Vector3d& d);                     // :139-143
    void set_fov(double fov) { fov_ = fov; }
    rt_camera to_pod() const;
    static Camera from_pod(const rt_camera& c);   // adopt already-derived vectors verbatim

private:
    algebra::Vector3d position_, direction_, up_, rigth_;
    double fov_, focal_length_;
};

}  // namespace camera

namespace world {

// src/world/ray.rs:5-18
struct Ray {
    algebra::Vector3d origin, direction;
    Ray() {}
    Ray(const algebra::Vector3d& o, const algebra::Vector3d& d) : origin(o), direction(d.normalize()) {}
};

// what Scene::closest_hit returns (RayHit, src/world/ray.rs:21-29) with the material reference
// replaced by the shape / material indices of the flat scene
struct RayHit {
    algebra::Vector3d point, normal;
    double distance;
    bool is_front_face;
    double u, v;
    int32_t shape_index;
};

// the flat structure-of-arrays copy of a Scene that crosses the C ABI
struct FlatScene {
    std::vector<uint8_t> kind, flags;
    std::vector<double> inverse, direct, params;
    std::vector<uint32_t> material;
    std::vector<rt_material> materials;
    std::vector<rt_texture> textures;
    std::vector<std::vector<uint8_t>> image_data;
    std::vector<rt_image> images;
    std::vector<rt_perlin> noise;
    std::vector<std::string> shape_names, material_names;
    rt_scene_desc desc() const;
};

// Image decoding hook standing in for `image::open` (src/world/texture.rs:128-139): returns RGBA8
// rows top-down or an empty vector.  Binary PPM (P6) is decoded natively; anything else goes to
// the registered loader (the Python package registers a PIL-based one).
typedef bool (*ImageLoaderFn)(const char* filename, uint32_t* width, uint32_t* height, uint8_t** rgba_malloced);
void set_image_loader(ImageLoaderFn fn);

// src/world/mod.rs:20-49 + src/world/json_models.rs:23-133
class Scene {
public:
    // Scene::from_json.  The reference appends ~481 random spheres from thread_rng on every load
    // (json_models.rs:44,50-133); `random_spheres_seed` makes that reproducible, and
    // `add_random_spheres = false` gives just the shapes in the file (for unit tests).
    // Throws std::runtime_error on malformed input (the reference returns serde_json::Error).
    static std::shared_ptr<Scene> from_json(const std::string& data, uint64_t random_spheres_seed = 1,
                                            bool add_random_spheres = true);
    ~Scene();

    const camera::Camera& camera() const { return camera_; }          // :193-196
    const FlatScene& flat() const { return flat_; }
    uint32_t shape_count() const { return (uint32_t)flat_.kind.size(); }

    // Re-point shape `shape_index` at the named material (used to build the config-4b variant
    // where every material / texture branch is live).  Must be called before the first device use.
    void assign_material(uint32_t shape_index, const std::string& material_name);

    // Move shapes: shape index[i] gets the InversableTransform whose rows 0..3 are direct16[16 i ..] and inverse16[16 i ..]
    // (row-major 4x4, as rth_transform_new gives them).  The description is edited and every device handle this scene
    // has created gets rt_scene_update_transforms, so that the scene and its handles stay in step.  Throws on a bad or
    // repeated index before anything changes; a handle that rejects the update (a frame in flight) throws after the
    // handles before it were updated.
    void set_transforms(uint32_t n, const uint32_t* index, const double* direct16, const double* inverse16);

    // Scene::closest_hit (:42-44) for a batch of rays — runs on the GPU.
    std::vector<RayHit> closest_hit(const std::vector<Ray>& rays, double min_t, double max_t,
                                    int mode = RT_ISECT_BRUTE, int device = 0);

    // the device-resident copy on `device` (created on first use, one per device, alive as long as the Scene)
    rt_scene* device_scene(int device = 0);
    // ONE handle over several devices (rt_scene_create_multi): whole-frame renders are sharded over all of them
    rt_scene* device_scene(const std::vector<int>& devices);

private:
    Scene() {}
    camera::Camera camera_;
    algebra::Vector3d background_;   // parsed, and ignored exactly like the reference (:199-202)
    FlatScene flat_;
    std::map<int, rt_scene*> dev_;
    std::map<std::vector<int>, rt_scene*> multi_;
};

}  // namespace world

namespace renderer {

// src/renderer/mod.rs:47-56
class Renderer {
public:
    virtual ~Renderer() {}
    virtual void start_rendering(std::shared_ptr<camera::Camera> camera, const camera::ImageParams& img_params,
                                 uint32_t samples_number) = 0;
    // true == frame complete; `buffer` (w*h, index x + y*w) is overwritten as pixels finish
    virtual bool render_step(std::vector<algebra::Vector3d>& buffer) = 0;
    virtual void stop_rendering() = 0;
};

// Drop-in for step_by_step::ThreadPoolRenderer (src/renderer/step_by_step.rs:37): same constructor
// convention (scene, thread_number, depth); thread_number is accepted and ignored (no CPU workers).
class GpuRenderer : public Renderer {
public:
    GpuRenderer(std::shared_ptr<world::Scene> scene, uint32_t thread_number, uint32_t depth, int device = 0,
                uint64_t seed = 0);
    // the same renderer over SEVERAL devices of the box (one process, one handle: rt_scene_create_multi); the frame
    // is the single-device one, bit for bit
    GpuRenderer(std::shared_ptr<world::Scene> scene, uint32_t thread_number, uint32_t depth,
                const std::vector<int>& devices, uint64_t seed = 0);
    void start_rendering(std::shared_ptr<camera::Camera> camera, const camera::ImageParams& img_params,
                         uint32_t samples_number) override;
    bool render_step(std::vector<algebra::Vector3d>& buffer) override;
    bool render_step(algebra::Vector3d* buffer, size_t len);   // same, on a raw caller-owned buffer
    void stop_rendering() override;

private:
    rt_scene* handle() const;
    std::shared_ptr<world::Scene> scene_;
    uint32_t depth_;
    int device_;
    std::vector<int> devices_;   // empty: the single device `device_`
    uint64_t seed_;
    bool started_;
    uint64_t pixels_;
};

}  // namespace renderer
}  // namespace ray_tracing
