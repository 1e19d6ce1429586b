//! `src/renderer/gpu.rs` (new file of the patch): the GPU drop-in for `step_by_step::ThreadPoolRenderer`
//! (src/renderer/step_by_step.rs:37-121) behind `pub trait Renderer` (src/renderer/mod.rs:47-56).
//! UNCOMPILED (no Rust toolchain in the authoring image); the tested equivalent is
//! `renderer::GpuRenderer` in rs_pathtracing_b200/csrc/host/ray_tracing.cpp.
use std::sync::{Arc, RwLock};

use ray_tracing_b200_sys as sys;

use crate::{
    algebra::Vector3d,
    camera::{ray_caster::ImageParams, Camera},
    renderer::Renderer,
    world::{flat::FlatScene, Scene},
};

fn v(a: &Vector3d) -> sys::rt_vec3 { sys::rt_vec3 { x: a.x, y: a.y, z: a.z } }
fn check(rc: i32) { if rc != sys::RT_OK { panic!("rt_b200: {}", sys::last_error()) } }  // the reference unwraps too

/// The reference renders whatever its `Arc<RwLock<Scene>>` holds when a frame starts (step_by_step.rs:37): the renderer
/// keeps the lock and, at every start_rendering, compares the flattened scene with what the device holds.
pub struct GpuRenderer {
    scene: *mut sys::rt_scene, depth: u32, seed: u64, progressive: bool,
    world: Arc<RwLock<Scene>>,
    uploaded: Vec<u8>,   // the bytes of the description the device holds (every table, images included)
}

/// every byte a description points at, in a fixed order: two descriptions give the same bytes iff they describe the
/// same scene
fn desc_bytes(d: &sys::rt_scene_desc) -> Vec<u8> {
    fn raw<T>(p: *const T, n: usize, out: &mut Vec<u8>) {
        if n > 0 && !p.is_null() {
            out.extend_from_slice(unsafe { std::slice::from_raw_parts(p as *const u8, n * std::mem::size_of::<T>()) });
        }
    }
    let n = d.n_shapes as usize;
    let mut out = Vec::new();
    out.extend_from_slice(&d.n_shapes.to_le_bytes());
    raw(d.kind, n, &mut out);
    raw(d.flags, n, &mut out);
    raw(d.inverse, 12 * n, &mut out);
    raw(d.direct, 12 * n, &mut out);
    raw(d.params, sys::RT_SHAPE_PARAMS as usize * n, &mut out);
    raw(d.material, n, &mut out);
    for (count, bytes) in [(d.n_materials, std::mem::size_of::<sys::rt_material>()),
                           (d.n_textures, std::mem::size_of::<sys::rt_texture>()),
                           (d.n_noise, std::mem::size_of::<sys::rt_perlin>())] {
        out.extend_from_slice(&count.to_le_bytes());
        out.extend_from_slice(&(bytes as u64).to_le_bytes());
    }
    raw(d.materials, d.n_materials as usize, &mut out);
    raw(d.textures, d.n_textures as usize, &mut out);
    raw(d.noise, d.n_noise as usize, &mut out);
    for i in 0..d.n_images as usize {
        let im = unsafe { &*d.images.add(i) };
        out.extend_from_slice(&im.width.to_le_bytes());
        out.extend_from_slice(&im.height.to_le_bytes());
        raw(im.rgba, 4 * im.width as usize * im.height as usize, &mut out);
    }
    out
}

impl GpuRenderer {
    /// same constructor convention as ThreadPoolRenderer::new (step_by_step.rs:37); `thread_number` is ignored
    pub fn new(scene: Arc<RwLock<Scene>>, thread_number: u32, depth: u32) -> Self {
        Self::with_devices(scene, thread_number, depth, &[0])
    }
    /// the same renderer over several GPUs of the box: ONE handle (rt_scene_create_multi), frames sharded by
    /// interleaved tiles over all of them, the assembled frame identical to the single-GPU one
    pub fn with_devices(scene: Arc<RwLock<Scene>>, _thread_number: u32, depth: u32, devices: &[i32]) -> Self {
        let (h, uploaded) = {
            let s = scene.read().unwrap();
            let f: &FlatScene = s.flat();
            let mut images = Vec::new();
            let desc = f.desc(&mut images);
            let mut h = std::ptr::null_mut();
            // (the library copies the description)
            check(unsafe { sys::rt_scene_create_multi(&desc, devices.len() as i32, devices.as_ptr(), &mut h) });
            (h, desc_bytes(&desc))
        };
        GpuRenderer { scene: h, depth, seed: 0, progressive: false, world: scene, uploaded }
    }
    /// Re-reads the RwLock'd scene and, when it differs from what the device holds, replaces the handle's scene in
    /// place (rt_scene_update: the handle keeps its streams, buffers and devices; the frame equals a fresh handle's).
    /// start_rendering calls it, so an edit made between two frames renders in the next one, as in the reference.
    pub fn sync_scene(&mut self) {
        let s = self.world.read().unwrap();
        let f: &FlatScene = s.flat();
        let mut images = Vec::new();
        let desc = f.desc(&mut images);
        let bytes = desc_bytes(&desc);
        if bytes != self.uploaded {
            check(unsafe { sys::rt_scene_update(self.scene, &desc) });
            self.uploaded = bytes;
        }
    }
    /// Progressive accumulation (rt_render_set_accumulate): while on, start_rendering calls with an unchanged
    /// camera ADD their samples to the frame instead of starting over -- what RendererState::render
    /// (main_raylib.rs:204-237) would call with samples_number = 1 per UI frame while the camera is still.
    pub fn set_progressive(&mut self, on: bool) {
        self.progressive = on;
        check(unsafe { sys::rt_render_set_accumulate(self.scene, on as i32) });
    }
}

impl Renderer for GpuRenderer {
    fn start_rendering(&mut self, camera: Arc<RwLock<Camera>>, img: &ImageParams, samples_number: u32) {
        self.stop_rendering();   // (rt_render_start stops a frame in flight too; the update must not meet one)
        self.sync_scene();
        let c = camera.read().unwrap();
        let cam = sys::rt_camera {
            position: v(c.position()), direction: v(c.direction()), up: v(c.up()), right: v(c.rigth()),
            fov_rad: c.fov(), focal_length: c.focal_length(),
        };
        let p = sys::rt_render_params {
            image: sys::rt_image_params { width: img.width, height: img.height },
            samples_number, max_depth: self.depth, seed: self.seed,
            shard_count: 1, shard_index: 0, tile_width: 0, tile_height: 0,
        };
        if !self.progressive { self.seed = self.seed.wrapping_add(1); } // a fresh stream per frame, like thread_rng
                                                                       // (an accumulating frame keeps its key)
        check(unsafe { sys::rt_render_start(self.scene, &cam, &p) });  // returns immediately
    }
    /// non-blocking, partial pixels may arrive before completion (step_by_step.rs:101-121);
    /// needs #[repr(C)] on algebra::Vector3d (3 x f64, src/algebra/mod.rs:23-28)
    fn render_step(&mut self, buffer: &mut Vec<Vector3d>) -> bool {
        let mut done = 0;
        check(unsafe { sys::rt_render_poll(self.scene, buffer.as_mut_ptr() as *mut sys::rt_vec3, &mut done) });
        done != 0
    }
    fn stop_rendering(&mut self) { check(unsafe { sys::rt_render_stop(self.scene) }); }
}

impl Drop for GpuRenderer { fn drop(&mut self) { unsafe { sys::rt_scene_destroy(self.scene) } } }
