/*
 * rt_b200_host.h — C shim over the C++ host-side mirror of the reference crate's interface
 * (rs_pathtracing_b200/csrc/host/ray_tracing.hpp), so that Python (ctypes) tests and tools can
 * drive the same code a C++ embedder links.  This is NOT the drop-in boundary (that is
 * rt_b200.h); it is the convenience layer above it:  Scene::from_json, Camera::new and the
 * GpuRenderer object that implements the Renderer trait.
 *
 * Reference interfaces mirrored (paths into dkarpushkin/rs-pathtracing):
 *   Scene::from_json                      src/world/mod.rs:46-49, src/world/json_models.rs:23-133
 *   Camera::new                           src/camera/mod.rs:71-88
 *   ThreadPoolRenderer::new / Renderer    src/renderer/step_by_step.rs:37, src/renderer/mod.rs:47-56
 */
#ifndef RT_B200_HOST_H
#define RT_B200_HOST_H

#include "rt_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rth_scene rth_scene;        /* std::shared_ptr<ray_tracing::world::Scene>      */
typedef struct rth_renderer rth_renderer;  /* ray_tracing::renderer::GpuRenderer              */

const char* rth_last_error(void);

/* image decoder hook standing in for image::open (src/world/texture.rs:128-139); the callee
 * returns malloc()ed RGBA8 rows, top row first */
typedef int (*rth_image_loader)(const char* filename, uint32_t* width, uint32_t* height, uint8_t** rgba);
void rth_set_image_loader(rth_image_loader fn);

/* Scene::from_json.  seed drives the reproducible stand-in for thread_rng in add_random_spheres
 * (json_models.rs:50-133); add_random_spheres = 0 loads only the shapes in the file. */
int rth_scene_from_json(const char* json_text, uint64_t random_spheres_seed, int add_random_spheres,
                        rth_scene** out);
void rth_scene_free(rth_scene* scene);
/* the flat description (pointers stay valid until rth_scene_free / rth_scene_assign_material) */
int rth_scene_desc(rth_scene* scene, rt_scene_desc* out);
int rth_scene_camera(rth_scene* scene, rt_camera* out);
uint32_t rth_scene_shape_count(rth_scene* scene);
const char* rth_scene_shape_name(rth_scene* scene, uint32_t index);
const char* rth_scene_material_name(rth_scene* scene, uint32_t index);
int rth_scene_assign_material(rth_scene* scene, uint32_t shape_index, const char* material_name);
/* Move shapes: shape index[i] gets the transform whose row-major 4x4 direct and inverse matrices are direct16[16 i ..] and
 * inverse16[16 i ..] (rth_transform_new's outputs).  Edits the description in place (rth_scene_desc pointers stay
 * valid) and applies rt_scene_update_transforms to every device handle the scene has created (rth_scene_device,
 * rth_scene_device_multi), so that the scene and its handles stay in step.  RT_ERR_INVALID for a NULL array with n > 0,
 * an index out of range or listed twice, before anything changes.  The handles are updated one after the other: when
 * one rejects the update (a frame in flight on it) the call fails, the handles before it were updated and the
 * description was not. */
int rth_scene_set_transforms(rth_scene* scene, uint32_t n, const uint32_t* index, const double* direct16,
                             const double* inverse16);
/* the device-resident rt_scene (uploaded on first use); owned by the rth_scene */
int rth_scene_device(rth_scene* scene, int device, rt_scene** out);
/* ONE rt_scene over several devices (rt_scene_create_multi), created on first use per device list */
int rth_scene_device_multi(rth_scene* scene, int n_devices, const int* device_ids, rt_scene** out);

/* Camera::new (fov in radians) */
int rth_camera_new(rt_vec3 position, rt_vec3 direction, rt_vec3 up, double focal_length, double fov_rad,
                   rt_camera* out);
/* InversableTransform::new: rows 0..3 of direct and inverse, row-major 4x4 */
int rth_transform_new(rt_vec3 translate, rt_vec3 rotate_deg, rt_vec3 scale, double* direct16, double* inverse16);

/* GpuRenderer: ThreadPoolRenderer::new(scene, thread_number, depth) + the Renderer trait */
int rth_renderer_new(rth_scene* scene, uint32_t thread_number, uint32_t depth, int device, uint64_t seed,
                     rth_renderer** out);
/* the same renderer over several devices of the box, one process (frames sharded by interleaved tiles) */
int rth_renderer_new_multi(rth_scene* scene, uint32_t thread_number, uint32_t depth, int n_devices,
                           const int* device_ids, uint64_t seed, rth_renderer** out);
void rth_renderer_free(rth_renderer* r);
int rth_renderer_start_rendering(rth_renderer* r, const rt_camera* camera, rt_image_params img,
                                 uint32_t samples_number);
/* *done = render_step's bool */
int rth_renderer_render_step(rth_renderer* r, rt_vec3* buffer, uint64_t buffer_len, int* done);
int rth_renderer_stop_rendering(rth_renderer* r);


/* image::save_buffer(path, &frame, w, h, ColorType::Rgba8) of the bins (src/bin/main_raylib.rs:64-75,
 * src/bin/main.rs:72-83): writes an 8-bit RGBA PNG (stored deflate blocks; no external library). */
int rth_save_png(const char* path, const uint8_t* rgba, uint32_t width, uint32_t height);

#ifdef __cplusplus
}
#endif
#endif
