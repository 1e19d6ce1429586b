//! Raw bindings to `include/rt_b200.h` (ABI version 5).  One item per declaration of the header; see
//! the header for the contract of every entry point and the reference interface it replaces.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const RT_B200_ABI_VERSION: c_int = 5;

// rt_status
pub const RT_OK: c_int = 0;
pub const RT_ERR_INVALID: c_int = -1;
pub const RT_ERR_NO_DEVICE: c_int = -2;
pub const RT_ERR_CUDA: c_int = -3;
pub const RT_ERR_STATE: c_int = -4;
pub const RT_ERR_NOMEM: c_int = -5;

// shape / surface / material / texture kinds
pub const RT_SHAPE_SPHERE: u8 = 0;
pub const RT_SHAPE_CUBE: u8 = 1;
pub const RT_SHAPE_RECTANGLE: u8 = 2;
pub const RT_SHAPE_MARCH: u8 = 3;
pub const RT_SHAPE_TORUS: u8 = 4;
pub const RT_SHAPE_FLAG_INVERSE_NORMAL: u8 = 1;
pub const RT_SHAPE_PARAMS: usize = 8;
pub const RT_SURF_HEART: u32 = 0;
pub const RT_SURF_SINE: u32 = 1;
pub const RT_SURF_STAR: u32 = 2;
pub const RT_SURF_DUPIN: u32 = 3;
pub const RT_SURF_HUNTS: u32 = 4;
pub const RT_SURF_CUSHION: u32 = 5;
pub const RT_MAT_LAMBERTIAN: u32 = 0;
pub const RT_MAT_METAL: u32 = 1;
pub const RT_MAT_DIELECTRIC: u32 = 2;
pub const RT_MAT_DIFFUSE_LIGHT: u32 = 3;
pub const RT_MAT_EMPTY: u32 = 4;
pub const RT_TEX_SOLID: u32 = 0;
pub const RT_TEX_CHECKER: u32 = 1;
pub const RT_TEX_UV_CHECKER: u32 = 2;
pub const RT_TEX_IMAGE: u32 = 3;
pub const RT_TEX_NOISE: u32 = 4;
pub const RT_ISECT_BRUTE: c_int = 0;
pub const RT_ISECT_FAST: c_int = 1;
pub const RT_ISECT_VERIFY: c_int = 2;
pub const RT_BOUNCE_MISS: u8 = 0;
pub const RT_BOUNCE_SCATTER: u8 = 1;
pub const RT_BOUNCE_EMIT: u8 = 2;

#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct rt_vec3 { pub x: f64, pub y: f64, pub z: f64 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_ray { pub origin: rt_vec3, pub direction: rt_vec3 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_camera {
    pub position: rt_vec3, pub direction: rt_vec3, pub up: rt_vec3, pub right: rt_vec3,
    pub fov_rad: f64, pub focal_length: f64 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_image_params { pub width: u32, pub height: u32 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_material { pub kind: u32, pub texture: u32, pub scalar: f64 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_texture {
    pub kind: u32, pub odd: u32, pub even: u32, pub image: u32, pub color: rt_vec3 }
#[repr(C)] pub struct rt_perlin {
    pub perm_x: [u32; 256], pub perm_y: [u32; 256], pub perm_z: [u32; 256], pub ranvec: [rt_vec3; 256] }
#[repr(C)] pub struct rt_image { pub width: u32, pub height: u32, pub rgba: *const u8 }
#[repr(C)] pub struct rt_scene_desc {
    pub n_shapes: u32, pub kind: *const u8, pub flags: *const u8,
    pub inverse: *const f64, pub direct: *const f64, pub params: *const f64, pub material: *const u32,
    pub n_materials: u32, pub materials: *const rt_material,
    pub n_textures: u32, pub textures: *const rt_texture,
    pub n_images: u32, pub images: *const rt_image,
    pub n_noise: u32, pub noise: *const rt_perlin }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_render_params {
    pub image: rt_image_params, pub samples_number: u32, pub max_depth: u32, pub seed: u64,
    pub shard_count: u32, pub shard_index: u32, pub tile_width: u32, pub tile_height: u32 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_adaptive_params {
    pub min_samples: u32, pub rel_error: f64, pub abs_error: f64 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct rt_feature_sums {
    pub albedo: rt_vec3, pub normal: rt_vec3, pub depth: f64, pub hits: f64, pub shape: i32, pub pad: u32 }
#[repr(C)] #[derive(Clone, Copy, Debug)] pub struct rt_feature_planes {
    pub albedo: *mut rt_vec3, pub normal: *mut rt_vec3, pub depth: *mut f64, pub coverage: *mut f64,
    pub shape: *mut i32 }
#[repr(C)] #[derive(Clone, Copy, Default, Debug)] pub struct rt_stats {
    pub kernel_launches: u64, pub paths: u64, pub segments: u64, pub shape_tests: u64, pub cull_tests: u64,
    pub march_steps: u64, pub march_rays: u64, pub march_long_rays: u64, pub march_max_evals: u64,
    pub last_frame_ms: f64, pub last_intersect_ms: f64, pub verify_rays: u64, pub verify_false_culls: u64,
    pub ms_raygen: f64, pub ms_extend: f64, pub ms_march: f64, pub ms_shade: f64, pub ms_resolve: f64,
    pub launches_extend: u64, pub launches_march: u64, pub launches_shade: u64, pub march_prof: [u64; 8] }
/// opaque: the device-resident scene + renderer state
pub enum rt_scene {}

extern "C" {
    pub fn rt_abi_version() -> c_int;
    pub fn rt_last_error() -> *const c_char;
    pub fn rt_device_count() -> c_int;
    pub fn rt_scene_create(desc: *const rt_scene_desc, device: c_int, out: *mut *mut rt_scene) -> c_int;
    pub fn rt_scene_destroy(scene: *mut rt_scene);
    pub fn rt_scene_create_multi(desc: *const rt_scene_desc, n_devices: c_int, device_ids: *const c_int,
        out: *mut *mut rt_scene) -> c_int;
    pub fn rt_scene_device_count(scene: *mut rt_scene) -> c_int;
    pub fn rt_scene_update(scene: *mut rt_scene, desc: *const rt_scene_desc) -> c_int;
    pub fn rt_scene_update_transforms(scene: *mut rt_scene, n: u32, shape_index: *const u32, inverse: *const f64,
        direct: *const f64) -> c_int;
    pub fn rt_intersect_batch(scene: *mut rt_scene, rays: *const rt_ray, n: u64, t_min: f64, t_max: f64,
        mode: c_int, shape_index: *mut i32, t: *mut f64, normal: *mut rt_vec3, point: *mut rt_vec3,
        uv: *mut f64, front_face: *mut u8) -> c_int;
    pub fn rt_intersect_batch_device(scene: *mut rt_scene, d_rays: *const rt_ray, n: u64, t_min: f64, t_max: f64,
        mode: c_int, d_shape_index: *mut i32, d_t: *mut f64, d_normal: *mut rt_vec3, d_point: *mut rt_vec3,
        d_uv: *mut f64, d_front_face: *mut u8, stream: *mut c_void) -> c_int;
    pub fn rt_occluded_batch(scene: *mut rt_scene, rays: *const rt_ray, n: u64, t_min: f64, t_max: f64,
        t_max_per_ray: *const f64, mode: c_int, occluded: *mut u8) -> c_int;
    pub fn rt_occluded_batch_device(scene: *mut rt_scene, d_rays: *const rt_ray, n: u64, t_min: f64, t_max: f64,
        d_t_max_per_ray: *const f64, mode: c_int, d_occluded: *mut u8, stream: *mut c_void) -> c_int;
    pub fn rt_scatter_batch(scene: *mut rt_scene, rays: *const rt_ray, keys: *const u32, n: u64, level: u32, seed: u64,
        t_min: f64, t_max: f64, mode: c_int, shape_index: *mut i32, t: *mut f64, outcome: *mut u8,
        color: *mut rt_vec3, scattered: *mut rt_ray) -> c_int;
    pub fn rt_scatter_batch_device(scene: *mut rt_scene, d_rays: *const rt_ray, d_keys: *const u32, n: u64,
        level: u32, seed: u64, t_min: f64, t_max: f64, mode: c_int, d_shape_index: *mut i32, d_t: *mut f64,
        d_outcome: *mut u8, d_color: *mut rt_vec3, d_scattered: *mut rt_ray, stream: *mut c_void) -> c_int;
    pub fn rt_render_start(scene: *mut rt_scene, camera: *const rt_camera, params: *const rt_render_params) -> c_int;
    pub fn rt_render_poll(scene: *mut rt_scene, buffer: *mut rt_vec3, done: *mut c_int) -> c_int;
    pub fn rt_render_wait(scene: *mut rt_scene, buffer: *mut rt_vec3) -> c_int;
    pub fn rt_render_stop(scene: *mut rt_scene) -> c_int;
    pub fn rt_render_set_accumulate(scene: *mut rt_scene, enabled: c_int) -> c_int;
    pub fn rt_render_accumulated_samples(scene: *mut rt_scene, samples: *mut u32) -> c_int;
    pub fn rt_render_start_adaptive(scene: *mut rt_scene, camera: *const rt_camera, params: *const rt_render_params,
        adaptive: *const rt_adaptive_params) -> c_int;
    pub fn rt_render_pixel_stats(scene: *mut rt_scene, counts: *mut u32, moments: *mut f64) -> c_int;
    pub fn rt_render_start_counts(scene: *mut rt_scene, camera: *const rt_camera, params: *const rt_render_params,
        counts: *const u32) -> c_int;
    pub fn rt_render_start_views(scene: *mut rt_scene, cameras: *const rt_camera, n_views: u32,
        params: *const rt_render_params) -> c_int;
    pub fn rt_render_start_layers(scene: *mut rt_scene, camera: *const rt_camera, params: *const rt_render_params,
        n_layers: u32) -> c_int;
    pub fn rt_render_layers(scene: *mut rt_scene, host: *mut rt_vec3, d_layers: *mut *const rt_vec3, n: *mut u64) -> c_int;
    pub fn rt_render_device_layers(scene: *mut rt_scene, d_sums: *mut *const rt_vec3, n_slots: *mut u64) -> c_int;
    pub fn rt_assemble_layers(scene: *mut rt_scene, params: *const rt_render_params, n_layers: u32,
        d_accs: *const *const c_void, d_layer_sums: *const *const c_void, d_out: *mut rt_vec3,
        stream: *mut c_void) -> c_int;
    pub fn rt_render_start_features(scene: *mut rt_scene, camera: *const rt_camera,
        params: *const rt_render_params) -> c_int;
    pub fn rt_render_features(scene: *mut rt_scene, host: *const rt_feature_planes,
        device: *mut rt_feature_planes) -> c_int;
    pub fn rt_render_device_features(scene: *mut rt_scene, d_sums: *mut *const rt_feature_sums,
        n_slots: *mut u64) -> c_int;
    pub fn rt_assemble_features(scene: *mut rt_scene, params: *const rt_render_params, d_sums: *const *const c_void,
        d_out: *const rt_feature_planes, stream: *mut c_void) -> c_int;
    pub fn rt_render_device_result(scene: *mut rt_scene, d_accum: *mut *const c_void, n_float4: *mut u64) -> c_int;
    pub fn rt_shard_float4_count(params: *const rt_render_params, shard_index: u32) -> u64;
    pub fn rt_assemble_frame(scene: *mut rt_scene, params: *const rt_render_params, d_shards: *const *const c_void,
        d_frame: *mut rt_vec3, stream: *mut c_void) -> c_int;
    pub fn rt_render_device_frame(scene: *mut rt_scene, d_frame: *mut *const rt_vec3, n_pixels: *mut u64) -> c_int;
    pub fn rt_tonemap_rgba8(scene: *mut rt_scene, frame: *const rt_vec3, n_pixels: u64, rgba: *mut u8) -> c_int;
    pub fn rt_tonemap_rgba8_device(scene: *mut rt_scene, d_rgba: *mut *const u8, rgba_host: *mut u8,
        n_pixels: *mut u64) -> c_int;
    pub fn rt_trace_pixel_samples(scene: *mut rt_scene, rays: *const rt_ray, n_rays: u32, max_depth: u32,
        seed: u64, pixel_index: u32, mean_out: *mut rt_vec3) -> c_int;
    pub fn rt_trace_pixel_samples_group(scene: *mut rt_scene, rays: *const rt_ray, n_rays: u64, offsets: *const u64,
        pixel_index: *const u32, n_groups: u32, max_depth: u32, seed: u64, means: *mut rt_vec3) -> c_int;
    pub fn rt_trace_pixel_samples_group_device(scene: *mut rt_scene, d_rays: *const rt_ray, n_rays: u64,
        offsets: *const u64, pixel_index: *const u32, n_groups: u32, max_depth: u32, seed: u64, d_means: *mut rt_vec3,
        stream: *mut c_void) -> c_int;
    pub fn rt_get_stats(scene: *mut rt_scene, out: *mut rt_stats) -> c_int;
    pub fn rt_reset_stats(scene: *mut rt_scene) -> c_int;
    pub fn rt_set_counters(scene: *mut rt_scene, enabled: c_int) -> c_int;
    pub fn rt_set_kernel_timing(scene: *mut rt_scene, enabled: c_int) -> c_int;
    pub fn rt_march_region_bounds(params8: *const f64, grad_bound: *mut f64, hess_bound: *mut f64) -> c_int;
    pub fn rt_advance_exact(a: f64, s: f64, m: i64, out: *mut f64) -> c_int;
    pub fn rt_div3_exact(a: *const f64, s: *const f64, n: u64, q: *mut f64) -> c_int;
    pub fn rt_march_candidates_host(params8: *const f64, inverse12: *const f64, rays: *const rt_ray, n: u64, t_min: f64,
                                    t_max: f64, best: f64, miss_proof: c_int, t_out: *mut f64, hit_out: *mut u8, evaluations: *mut u64) -> c_int;
    pub fn rt_bernstein_clear(coefficients: *const f64, degree: c_int, length: f64, threshold: f64, clear: *mut c_int) -> c_int;
    pub fn rt_cull_reached(desc: *const rt_scene_desc, rays: *const rt_ray, n_rays: u64, reached: *mut u8) -> c_int;
    pub fn rt_cull_tree_check(desc: *const rt_scene_desc, n_roots: *mut u32, n_groups: *mut u32, n_tree: *mut u32,
        n_flat: *mut u32, worst: *mut f64) -> c_int;
    pub fn rt_cull_refit_check(desc: *const rt_scene_desc, n: u32, shape_index: *const u32, inverse: *const f64,
        worst: *mut f64) -> c_int;
    pub fn rt_measure_peaks(device: c_int, fp64_tflops: *mut f64, fp32_tflops: *mut f64) -> c_int;
}

/// `rt_last_error()` as an owned string
pub fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(rt_last_error()).to_string_lossy().into_owned() }
}
