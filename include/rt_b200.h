/*
 * rt_b200.h — C ABI of the B200-native path-tracing core for rs-pathtracing.
 *
 * This is the drop-in boundary: everything the Rust crate's FFI (`-sys` crate whose
 * build.rs runs nvcc) would bind for the hot path.  Plain C, plain pointers and sizes,
 * no C++ / torch types.  All `path:line` citations are into the reference repository
 * (dkarpushkin/rs-pathtracing).
 *
 * The reference has no FFI layer of its own; the seam that this ABI sits under is
 *   pub trait Renderer { start_rendering, render_step, stop_rendering }   src/renderer/mod.rs:47-56
 *   ThreadPoolRenderer::new(scene, thread_number, depth)                  src/renderer/step_by_step.rs:37
 *   Scene::closest_hit(&Ray, min_t, max_t)                                src/world/mod.rs:42-44
 *   renderer::trace_pixel_samples(&(idx, rays), &Scene, depth)            src/renderer/mod.rs:151-155
 *   renderer::trace_pixel_samples_group(&[(idx, rays)], &Scene, depth)    src/renderer/mod.rs:127-149
 *
 * Conventions
 *   - every entry point returns 0 (RT_OK) or a negative rt_status; nothing unwinds or aborts
 *     across the boundary; rt_last_error() gives the message of the calling thread's last failure.
 *   - the caller owns every host buffer; the library owns every device buffer unless a
 *     function is documented as taking a caller-supplied DEVICE pointer.
 *   - handles are not thread-safe (the reference calls the Renderer from one UI thread).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     RT_ERR_NO_DEVICE.
 */
#ifndef RT_B200_H
#define RT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_B200_ABI_VERSION 5

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID = -1,    /* bad argument / malformed scene description            */
    RT_ERR_NO_DEVICE = -2,  /* no CUDA device (the product path never falls back)     */
    RT_ERR_CUDA = -3,       /* a CUDA runtime call failed; see rt_last_error()        */
    RT_ERR_STATE = -4,      /* call out of order (poll without start, ...)            */
    RT_ERR_NOMEM = -5
} rt_status;

/* ---- POD mirrors of the reference's algebra / camera types ------------------------- */

/* algebra::Vector3d, src/algebra/mod.rs:23-28 (needs a #[repr(C)] mirror on the Rust side) */
typedef struct rt_vec3 { double x, y, z; } rt_vec3;

/* world::ray::Ray, src/world/ray.rs:5-9.  `direction` is what Ray::new produced (unit length,
 * ray.rs:12-17); the library never renormalises a caller-supplied ray. */
typedef struct rt_ray { rt_vec3 origin, direction; } rt_ray;

/* camera::Camera after Camera::new, src/camera/mod.rs:36-46,71-88:
 * direction/up/right are the derived unit vectors, fov in RADIANS. */
typedef struct rt_camera {
    rt_vec3 position, direction, up, right;
    double fov_rad, focal_length;
} rt_camera;

/* camera::ray_caster::ImageParams, src/camera/ray_caster.rs:10-14 */
typedef struct rt_image_params { uint32_t width, height; } rt_image_params;

/* ---- flat scene description (structure of arrays) ---------------------------------- */

/* Shape::ray_intersect implementations on the hot path, src/world/shapes/mod.rs:181,250,330 and
 * src/world/shapes/ray_marching.rs:20 */
enum {
    RT_SHAPE_SPHERE = 0,     /* unit sphere, flag bit0 = inverse_normal                         */
    RT_SHAPE_CUBE = 1,       /* unit box [-1,1]^3                                               */
    RT_SHAPE_RECTANGLE = 2,  /* z = 0 plane clipped to [x0,x1]x[y0,y1]; params = x0,y0,x1,y1    */
    RT_SHAPE_MARCH = 3,      /* RayMarchingShape; params below                                  */
    RT_SHAPE_TORUS = 4       /* Torus (src/world/shapes/mod.rs:403-494): params = radius, tube_radius; quartic via
                                the reference's complex Ferrari solver (src/algebra/equation.rs:17-67).  A root
                                counts as real when |im| < 1e-15, which depends on the last ulp of libm's
                                hypot / atan2 / cos / sin / cbrt: t agrees with the oracle to ~1e-12 relative where
                                both accept the root, the accept / reject decision itself is not bit-reproducible
                                across math libraries (neither is it between two builds of the reference)          */
};
#define RT_SHAPE_FLAG_INVERSE_NORMAL 1u

/* ShapeFunction implementations, src/world/shapes/ray_marching.rs:121-520 */
enum {
    RT_SURF_HEART = 0,   /* bound: ellipsoid radii (1.45, 1.45/2.05, 1.45)                      */
    RT_SURF_SINE = 1,    /* params a, sphere_radius                                              */
    RT_SURF_STAR = 2,    /* params a, sphere_radius                                              */
    RT_SURF_DUPIN = 3,   /* params a, b, c, d, sphere_radius                                     */
    RT_SURF_HUNTS = 4,   /* params sphere_radius                                                 */
    RT_SURF_CUSHION = 5  /* params sphere_radius                                                 */
};

/* params[i][8] layout
 *   RECTANGLE: [0]=x0 [1]=y0 [2]=x1 [3]=y1
 *   MARCH:     [0]=surface kind (as double) [1]=step [2]=depth (as double, u8 in the reference)
 *              [3]=a [4]=b [5]=c [6]=d [7]=sphere_radius
 *   SPHERE/CUBE: unused (zero)
 */
#define RT_SHAPE_PARAMS 8

/* Material implementations, src/world/material.rs:36-134 */
enum {
    RT_MAT_LAMBERTIAN = 0,   /* texture = albedo                       */
    RT_MAT_METAL = 1,        /* texture = albedo, scalar = fuzz        */
    RT_MAT_DIELECTRIC = 2,   /* scalar = index_of_refraction           */
    RT_MAT_DIFFUSE_LIGHT = 3,/* texture = emit                         */
    RT_MAT_EMPTY = 4
};
typedef struct rt_material {
    uint32_t kind;
    uint32_t texture;   /* index into textures[] (ignored for DIELECTRIC / EMPTY) */
    double scalar;
} rt_material;

/* Texture implementations, src/world/texture.rs:10-117 */
enum {
    RT_TEX_SOLID = 0,      /* color                                                   */
    RT_TEX_CHECKER = 1,    /* color = multipliers (x,y,z); odd/even texture indices   */
    RT_TEX_UV_CHECKER = 2, /* color.x/.y = multipliers .0/.1; odd/even                */
    RT_TEX_IMAGE = 3,      /* image = index into images[]                             */
    RT_TEX_NOISE = 4       /* NoiseTexture (texture.rs:54-68): image = index into noise[], color.x = scale */
};
typedef struct rt_texture {
    uint32_t kind;
    uint32_t odd, even;   /* child texture indices, in any order of the table.  Textures may share children, but
                             the graph must be acyclic, and no path down from a texture may cross more than
                             RT_TEX_MAX_DEPTH checker (CHECKER / UV_CHECKER) nodes before its leaf: 8 checkers
                             above a leaf are accepted, 9 are RT_ERR_INVALID */
    uint32_t image;
    rt_vec3 color;
} rt_texture;
#define RT_TEX_MAX_DEPTH 8

/* algebra::noise::Perlin (src/algebra/noise.rs:7-15): the tables Perlin::new draws from thread_rng
 * (:24-41) -- three permutations of 0..255 and 256 vectors with components in [-1, 1).  `ranfloat`
 * and `cartesian` are not used by noise() / turb() and are not carried. */
typedef struct rt_perlin {
    uint32_t perm_x[256], perm_y[256], perm_z[256];
    rt_vec3 ranvec[256];
} rt_perlin;

/* image::RgbaImage, row-major, 4 bytes per texel, row 0 = top (src/world/texture.rs:98-117) */
typedef struct rt_image {
    uint32_t width, height;
    const uint8_t* rgba;
} rt_image;

typedef struct rt_scene_desc {
    uint32_t n_shapes;
    const uint8_t* kind;        /* [n_shapes]                                                   */
    const uint8_t* flags;       /* [n_shapes]                                                   */
    const double* inverse;      /* [n_shapes][12]: rows 0..2 of InversableTransform.inverse     */
    const double* direct;       /* [n_shapes][12]: rows 0..2 of InversableTransform.direct      */
    const double* params;       /* [n_shapes][RT_SHAPE_PARAMS]                                  */
    const uint32_t* material;   /* [n_shapes] index into materials[]                            */
    uint32_t n_materials;
    const rt_material* materials;
    uint32_t n_textures;
    const rt_texture* textures;
    uint32_t n_images;
    const rt_image* images;
    uint32_t n_noise;
    const rt_perlin* noise;     /* [n_noise] Perlin tables of the NoiseTextures                 */
} rt_scene_desc;

typedef struct rt_scene rt_scene;   /* opaque: the device-resident scene + renderer state */

/* ---- library ------------------------------------------------------------------------ */

int rt_abi_version(void);
const char* rt_last_error(void);
/* number of visible CUDA devices (0 on a CPU-only host; never fails) */
int rt_device_count(void);

/* ---- scene -------------------------------------------------------------------------- */

/* Upload a flattened Scene to `device` (replaces Arc<RwLock<Scene>> handed to
 * ThreadPoolRenderer::new, src/renderer/step_by_step.rs:37).  The description is copied;
 * the caller may free it afterwards.
 * The description is checked before any device is touched (so RT_ERR_INVALID comes before RT_ERR_NO_DEVICE;
 * rt_scene_create_multi and rt_cull_tree_check apply the same check).  RT_ERR_INVALID when:
 *   - a table with a non-zero count is NULL (shape arrays, materials, textures, images, noise);
 *   - a kind is unknown, or a shape's material, a material's texture, a texture's child, image or noise index is
 *     out of range;
 *   - the texture graph has a cycle, or a path of more than RT_TEX_MAX_DEPTH checker nodes (see rt_texture);
 *   - a Perlin permutation entry (perm_x / perm_y / perm_z) is 256 or more;
 *   - an image has no pixels, no data, or more than SIZE_MAX / 4 texels (4 * width * height bytes must be
 *     addressable). */
int rt_scene_create(const rt_scene_desc* desc, int device, rt_scene** out);
void rt_scene_destroy(rt_scene* scene);

/* The same for SEVERAL devices of one box behind ONE handle -- what a single-process caller like the reference's
 * bins (one UI thread, one `impl Renderer`, src/renderer/mod.rs:47-56) needs to use more than one GPU.  The scene
 * is replicated on every listed device.  A whole-frame rt_render_start (shard_count 0 or 1) is then sharded over
 * the devices by interleaved tiles (the rule documented at rt_render_params, shard k on device_ids[k]); the shards
 * render concurrently, each accumulator reaches device_ids[0] with one peer copy on its own stream, and the frame
 * is assembled there.  rt_render_poll / rt_render_wait deliver the assembled frame (no partial delivery: *done
 * flips when the whole frame is there), rt_render_device_frame exposes it on device_ids[0].  The frame is the one a
 * single device renders, bit for bit (the RNG is keyed per pixel, the accumulators are f64 sums).  Every other
 * entry point (rt_intersect_batch, rt_trace_pixel_samples[_group], statistics, an explicitly sharded rt_render_start)
 * addresses device_ids[0].  n_devices = 1 is rt_scene_create. */
int rt_scene_create_multi(const rt_scene_desc* desc, int n_devices, const int* device_ids, rt_scene** out);
/* number of devices behind the handle (1 for rt_scene_create) */
int rt_scene_device_count(rt_scene* scene);

/* ---- batched nearest hit (replaces Scene::closest_hit, src/world/mod.rs:42-44, with the
 *      ShapeCollection semantics of src/world/shapes/mod.rs:573-597) -------------------- */

/* mode for rt_intersect_batch */
enum {
    RT_ISECT_BRUTE = 0,   /* one thread per ray walks the whole shape list in index order: the
                             literal restatement of ShapeCollection::ray_intersect             */
    RT_ISECT_FAST = 1,    /* conservative culling + exact FP64 test on the survivors; provably the
                             same result as RT_ISECT_BRUTE (degenerate rays fall back to it)     */
    RT_ISECT_VERIFY = 2   /* self-check: runs FAST and BRUTE on every ray, returns BRUTE's result and
                             counts disagreements + falsely culled (ray, shape) pairs in rt_stats   */
};

/* Host buffers in, host buffers out.  Any output pointer may be NULL.
 *   shape_index[i] = winning shape, -1 = miss
 *   t[i]           = RayHit.distance
 *   normal[i]      = RayHit.normal() after set_normal (unit, facing the ray), world space
 *   point[i]       = RayHit.point (direct transform of the object-space hit point)
 *   uv[2i..2i+1]   = RayHit.u, RayHit.v
 *   front_face[i]  = RayHit.is_front_face
 */
int rt_intersect_batch(rt_scene* scene, const rt_ray* rays, uint64_t n, double t_min, double t_max,
                       int mode, int32_t* shape_index, double* t, rt_vec3* normal, rt_vec3* point,
                       double* uv, uint8_t* front_face);

/* Same, with every pointer a DEVICE pointer on the scene's device and no copies; runs on
 * `stream` (a cudaStream_t passed as void*, NULL = the library's own non-blocking stream; the legacy
 * default stream, whose handle is 0, is named by cudaStreamLegacy = 0x1) and does not
 * synchronise.  Used for kernel-only timing and by callers that keep rays resident. */
int rt_intersect_batch_device(rt_scene* scene, const rt_ray* d_rays, uint64_t n, double t_min,
                              double t_max, int mode, int32_t* d_shape_index, double* d_t,
                              rt_vec3* d_normal, rt_vec3* d_point, double* d_uv,
                              uint8_t* d_front_face, void* stream);

/* ---- frame rendering (replaces the Renderer trait, src/renderer/mod.rs:47-56) -------- */

typedef struct rt_render_params {
    rt_image_params image;
    uint32_t samples_number;   /* start_rendering's samples_number                               */
    uint32_t max_depth;        /* ThreadPoolRenderer::new's depth (ray_color's depth argument); at most 62 */
    uint64_t seed;             /* counter-based RNG key                                          */
    /* image sharding (one process per GPU): this handle renders the tiles k with k % shard_count == shard_index.
     * 1 / 0 = whole image.  Tile NUMBERING (shard_count > 1): with tiles_x = ceil(width / tile_width), tile
     * number k lies in tile row ty = k / tiles_x at tile column
     *     tx = (k % tiles_x + ty % tiles_x) % tiles_x
     * -- row-major, with row ty rotated by ty positions, so that a shard owns diagonals instead of whole columns
     * of tiles when tiles_x is a multiple of shard_count.  A shard's accumulator (rt_render_device_result) lists
     * its tiles in increasing k, each tile row-major and padded to tile_width*tile_height at the image border.
     * rt_assemble_frame is the supported way to turn gathered accumulators back into a frame. */
    uint32_t shard_count, shard_index;
    uint32_t tile_width, tile_height;   /* 0 = default (32 x 32); tile_width * tile_height must be below 2^32
                                           (RT_ERR_INVALID from rt_render_start / rt_assemble_frame, and
                                           rt_shard_float4_count returns 0, otherwise)                        */
} rt_render_params;

/* Renderer::start_rendering: returns immediately, work proceeds on the library's stream. */
int rt_render_start(rt_scene* scene, const rt_camera* camera, const rt_render_params* params);

/* Renderer::render_step: non-blocking.  Writes the pixels finished so far into
 * buffer[x + y*width] (linear per-pixel mean radiance, src/renderer/mod.rs:151-155; pixels of
 * other shards are left untouched) and sets *done to 1 when the frame (this shard) is
 * complete, exactly like render_step's bool. */
int rt_render_poll(rt_scene* scene, rt_vec3* buffer, int* done);

/* Blocking convenience: waits for completion, then behaves like a final rt_render_poll. */
int rt_render_wait(rt_scene* scene, rt_vec3* buffer);

/* Renderer::stop_rendering: abandons the frame in flight (no-op when idle). */
int rt_render_stop(rt_scene* scene);

/* Progressive accumulation across rt_render_start calls (SURVEY 8f-3; the reference's interactive loop,
 * src/bin/main_raylib.rs:204-237, re-renders from scratch every time).  While enabled, a frame started with
 * the same camera, image, sharding, max_depth and seed as the previous one ADDS its samples_number samples to
 * the accumulator: its paths take the sample indices that follow the ones already traced (so k frames of n
 * samples are the very paths of one frame of k*n samples), and rt_render_poll / rt_render_device_result deliver
 * the mean over everything accumulated, bit for bit).  Any other frame, and every call of this function, starts
 * afresh.  Scenes with more than 32 ray-marched shapes are rendered by the fused fallback kernel, which cannot
 * accumulate: enabling returns RT_ERR_STATE there.
 * rt_render_accumulated_samples: the number of samples per pixel the accumulator holds (0 = empty). */
int rt_render_set_accumulate(rt_scene* scene, int enabled);
int rt_render_accumulated_samples(rt_scene* scene, uint32_t* samples);

/* Adaptive sampling: per-pixel sample counts driven by a noise target.  Every pixel of an adaptive frame equals, bit for
 * bit, what rt_render_start (or rt_trace_pixel_samples over the camera's primary rays) gives for that pixel at the
 * sample count it ended with; only the choice of that count is new.
 *   Luminance of a sample: y = (0.2126*r + 0.7152*g) + 0.0722*b of the path's float radiance widened to double, in that
 *   order, without FMA.  Σy and Σy² are f64 sums in sample order, kept per pixel next to the rgb sums.
 *   Schedule: pass 0 gives every pixel min_samples samples.  At each pass boundary, a pixel traced in the previous pass
 *   holding n samples is tested; it continues when it is not converged and n < samples_number, with
 *   m = min(n, samples_number - n) more samples numbered n .. n+m-1.  A pixel that stops is never tested again.  So
 *   the counts lie in {min_samples * 2^j} and {samples_number}.
 *   Stopping rule (in this operation order):
 *       mean = Sy / n
 *       var  = fmax(0, (Syy - Sy*mean) / (n-1))
 *       se   = sqrt(var / n)
 *       converged  iff  se <= fmax(rel_error * fabs(mean), abs_error)
 *   Consequences: min_samples == samples_number (or a huge rel_error) gives the rt_render_start frame bit for bit, plus
 *   its moments.  The result does not depend on the batch size, the lanes or the order in which pixels are listed:
 *   every decision is a function of a pixel's own bit-exact sums.  Stopping on the samples themselves biases the frame
 *   slightly, as any variance-driven sampler does (a pixel whose first samples missed a rare bright path stops early);
 *   each pixel is still exactly the reference's trace_pixel_samples of its own camera rays. */
typedef struct rt_adaptive_params {
    uint32_t min_samples;   /* every pixel gets these; 2 <= min_samples <= samples_number                   */
    double rel_error;       /* target standard error of the mean luminance, relative to the mean (>= 0)     */
    double abs_error;       /* absolute floor of that target (>= 0); both finite                            */
} rt_adaptive_params;

/* Starts an adaptive frame of at most params->samples_number samples per pixel.  Non-blocking like rt_render_start (a
 * frame in flight is stopped first): the whole frame is enqueued at once and runs without host synchronisation.
 * rt_render_poll reports done = 0 and leaves the buffer alone until the last pass has resolved, then delivers the whole
 * frame; rt_render_wait, rt_render_stop, rt_render_device_frame, rt_render_device_result and rt_tonemap_rgba8_device
 * work on the result.  The frame never continues or seeds a progressive accumulation (rt_render_accumulated_samples
 * reads 0 after it); rt_stats.paths grows by the sum of the counts once the frame is complete.
 * RT_ERR_INVALID: a multi-device handle, shard_count > 1, or bad parameters.  RT_ERR_STATE: a scene with more than 32
 * ray-marched shapes (the fused fallback renders it), as for rt_render_set_accumulate. */
int rt_render_start_adaptive(rt_scene* scene, const rt_camera* camera, const rt_render_params* params,
                             const rt_adaptive_params* adaptive);
/* After a completed unsharded single-device frame (adaptive or not; waits for the frame in flight), per pixel x + y*width:
 * counts[p] = the samples the pixel holds, moments[2p], moments[2p+1] = Σy, Σy² (adaptive frames only: RT_ERR_STATE
 * otherwise).  Either output may be NULL. */
int rt_render_pixel_stats(rt_scene* scene, uint32_t* counts, double* moments);

/* Device-side result of the last started frame, for callers that gather shards over NCCL:
 * FOUR DOUBLES (r, g, b sums; samples) per owned pixel -- the f64 sums themselves, so that the assembled frame
 * equals the unsharded one bit for bit; they were floats before ABI 4, hence the names -- tile-packed in this
 * shard's tile order (see rt_render_params; tiles clipped at the image border are still padded to
 * tile_width*tile_height).  *d_accum is a device pointer owned by the library, valid until the
 * next rt_render_start / rt_scene_destroy; *n_float4 the number of 4-vectors.  The frame must be complete. */
int rt_render_device_result(rt_scene* scene, const void** d_accum, uint64_t* n_float4);

/* number of 4-vector slots (32 bytes each) a shard owns, so every rank can size the gather */
uint64_t rt_shard_float4_count(const rt_render_params* params, uint32_t shard_index);

/* The completed frame on the device: *d_frame = width*height rt_vec3 (x + y*width, linear mean radiance) on the
 * handle's (first) device, valid until the next rt_render_start; waits for the frame in flight.  For an unsharded
 * frame of a single-device handle and for every frame of a multi-device handle. */
int rt_render_device_frame(rt_scene* scene, const rt_vec3** d_frame, uint64_t* n_pixels);

/* Assemble a full frame from the gathered shard buffers (all DEVICE pointers on the scene's
 * device): d_shards[s] = shard s's tile-packed float4 buffer; d_frame = w*h rt_vec3 (x + y*w,
 * linear mean).  Runs on `stream`, does not synchronise.  NULL = the library's own non-blocking stream, which is
 * NOT ordered against the caller's copies / NCCL receives into d_shards: a caller whose stream is the legacy
 * default stream (handle 0, e.g. torch's default stream) passes cudaStreamLegacy (0x1) to name it. */
int rt_assemble_frame(rt_scene* scene, const rt_render_params* params, const void* const* d_shards,
                      rt_vec3* d_frame, void* stream);

/* Frame post-process of the bins (src/bin/main_raylib.rs:239-247): sqrt, clamp(0,0.999)*256 ->
 * RGBA8, alpha 255.  Host in / host out convenience running on the device (persistent device buffers). */
int rt_tonemap_rgba8(rt_scene* scene, const rt_vec3* frame, uint64_t n_pixels, uint8_t* rgba);
/* The same applied to the frame the library already holds on the device (rt_render_device_frame): no f64 frame
 * crosses the bus -- 4 bytes per pixel instead of 24 come back.  Either output may be NULL: *d_rgba = the
 * library's persistent RGBA8 buffer on the device (valid until the next tonemap call), rgba_host = a host buffer
 * of 4*n_pixels bytes to copy it to. */
int rt_tonemap_rgba8_device(rt_scene* scene, const uint8_t** d_rgba, uint8_t* rgba_host, uint64_t* n_pixels);

/* ---- pixel probe (replaces renderer::trace_pixel_samples, src/renderer/mod.rs:151-155) */

/* Traces caller-supplied primary rays (host buffer) as samples of ONE pixel and returns their
 * mean radiance; RNG keyed by (seed, pixel_index, sample = ray number).  The one-group case of
 * rt_trace_pixel_samples_group; n_rays = 0 is rejected. */
int rt_trace_pixel_samples(rt_scene* scene, const rt_ray* rays, uint32_t n_rays, uint32_t max_depth,
                           uint64_t seed, uint32_t pixel_index, rt_vec3* mean_out);

/* renderer::trace_pixel_samples_group, src/renderer/mod.rs:127-149: many pixels in one wavefront.
 * Group g is rays[offsets[g] .. offsets[g+1]), samples 0, 1, ... of pixel pixel_index[g]; means[g] = the sum of
 * their ray_color / n_g with the arithmetic of rt_trace_pixel_samples (RNG keyed by (seed, pixel_index[g], sample),
 * per-path radiance rounded to float, f64 sum in sample order, one division).  So group g gives what
 * rt_trace_pixel_samples gives for its rays alone, and the camera's own primary rays with pixel_index = x + y*width
 * give the pixels of the rt_render_start frame of the same seed, depth and samples -- bit for bit, whatever the
 * batch size, the lanes, the order of the groups or their split into calls.  An empty group gives NaN (the
 * reference's Vector3d / 0.0); pixel indices may repeat; rays are never renormalised; n_groups = 0 does nothing.
 * RT_ERR_INVALID: offsets[0] != 0, decreasing offsets, offsets[n_groups] != n_rays, a group of 2^32 rays or more,
 * a NULL array that is needed, max_depth > 62.  RT_ERR_STATE while a frame is in flight.  The frame, its
 * accumulator and the progressive accumulation are left alone; rt_stats.paths grows by n_rays.  Addresses
 * device_ids[0] of a multi-device handle.  Blocks until means[] is written. */
int rt_trace_pixel_samples_group(rt_scene* scene, const rt_ray* rays, uint64_t n_rays,
                                 const uint64_t* offsets /* n_groups + 1 */, const uint32_t* pixel_index /* n_groups */,
                                 uint32_t n_groups, uint32_t max_depth, uint64_t seed, rt_vec3* means /* n_groups */);
/* The same with d_rays and d_means DEVICE pointers on the scene's (first) device; offsets and pixel_index stay HOST
 * arrays (the batches are planned from them; they are read before the call returns, pinned or pageable).  Ordered after the work queued
 * on `stream` before the call, and work queued on `stream` after it runs after d_rays has been read and d_means
 * written; returns without waiting (except while rt_set_kernel_timing is on).  stream: a cudaStream_t as void*;
 * NULL = the library's own non-blocking stream; the legacy default stream (handle 0, e.g. torch's default stream) is
 * named by cudaStreamLegacy = 0x1. */
int rt_trace_pixel_samples_group_device(rt_scene* scene, const rt_ray* d_rays, uint64_t n_rays,
                                        const uint64_t* offsets, const uint32_t* pixel_index, uint32_t n_groups,
                                        uint32_t max_depth, uint64_t seed, rt_vec3* d_means, void* stream);

/* ---- instrumentation ---------------------------------------------------------------- */

typedef struct rt_stats {
    uint64_t kernel_launches;   /* kernels launched by the library since the last reset         */
    uint64_t paths;             /* primary paths started                                        */
    uint64_t segments;          /* ray segments traced (nearest-hit queries)                    */
    uint64_t shape_tests;       /* exact FP64 shape tests executed                              */
    uint64_t cull_tests;        /* conservative pre-tests executed                              */
    uint64_t march_steps;       /* implicit-surface function evaluations                        */
    uint64_t march_rays;        /* (ray, marching shape) pairs marched                          */
    uint64_t march_long_rays;   /* ... of which needed more than 2048 evaluations               */
    uint64_t march_max_evals;   /* most evaluations a single marched ray needed                 */
    double last_frame_ms;       /* device time of the last completed frame (CUDA events)        */
    double last_intersect_ms;   /* device time of the last rt_intersect_batch kernel            */
    uint64_t verify_rays;        /* RT_ISECT_VERIFY: rays whose FAST result differs from BRUTE   */
    uint64_t verify_false_culls; /* RT_ISECT_VERIFY: culled (ray, shape) pairs the exact test hits */
    /* device time per kernel class since the last reset, summed over launches (CUDA event pairs on
     * the library's stream; only while rt_set_kernel_timing is on) and the launches they cover */
    double ms_raygen, ms_extend, ms_march, ms_shade, ms_resolve;
    uint64_t launches_extend, launches_march, launches_shade;
    /* k_march work breakdown (with counters on): literal steps at level 0, literal steps at the
     * refinement levels, exact multi-step jumps, hops of the skip bound, rays proven to miss by the Bernstein hull
     * of the surface polynomial / by the hop loop (no marching at all), plans that found nothing to skip at level 0 /
     * at a refinement level.  8 entries since ABI 5 (4 before) */
    uint64_t march_prof[8];
} rt_stats;
int rt_get_stats(rt_scene* scene, rt_stats* out);
int rt_reset_stats(rt_scene* scene);
/* enable (1) / disable (0) the per-kernel work counters above (segments..march_rays); counting
 * costs a few atomics per block and is off by default.  kernel_launches / *_ms are always on. */
int rt_set_counters(rt_scene* scene, int enabled);
/* enable (1) / disable (0) per-kernel device timing (rt_stats.ms_*): one CUDA event pair around every
 * launch of the following frames.  Not allowed while a frame is in flight. */
int rt_set_kernel_timing(rt_scene* scene, int enabled);

/* Host-only helper behind the exact-skip marcher: rigorous interval bounds G >= sup |grad f| and
 * H >= sup |u^T Hess f u| of a ray-marched surface (params8 = the shape's params row) over its marching
 * region.  Exposed so that tests can check them against sampled derivatives; needs no device. */
int rt_march_region_bounds(const double* params8, double* grad_bound, double* hess_bound);

/* Host-only build of the marcher's exact multi-step advance (csrc/rt_march.cuh, advance_exact): *out = the
 * double `a` holds after m iterations of `a = a + s` (IEEE round-to-nearest-even), computed in
 * O(binades crossed) like on the device.  Exposed so that CPU tests can compare it with the literal loop. */
int rt_advance_exact(double a, double s, int64_t m, double* out);

/* Host-only build of the device's vector / scalar division (csrc/rt_math.cuh, div3_exact): the three quotients
 * a[k] / s from one correctly rounded reciprocal and two FMA correction steps each.  q[3n] receives, for every
 * triple a[3i..3i+2] and divisor s[i], what the device computes; CPU tests compare it bit for bit with the IEEE
 * divisions the reference performs (Vector3d / f64, src/algebra/mod.rs:299-317).  Needs no device. */
int rt_div3_exact(const double* a, const double* s, uint64_t n, double* q);

/* Host-only build of the WHOLE exact-skip marcher (csrc/rt_march.cuh: Marcher -- the miss proof, jump planning, the
 * exact multi-step advance, landing self-check, literal steps, the local model of the refinement levels), the very
 * source the kernels compile: for one ray-marched shape (params8 = its rt_scene_desc params row, inverse12 = rows 0..2
 * of its inverse transform) and n world-space rays, the candidate RayMarchingShape::ray_intersect returns
 * (src/world/shapes/ray_marching.rs:20-74) with the chord clipped at best + 2 steps like k_march does (best = +inf:
 * unclipped).  miss_proof != 0: with the Bernstein-hull miss proof at the start of the ray, as k_march_filter runs it
 * (the per-lane device callers leave it out).  hit_out[i] = 1 and t_out[i] = t, or 0.  evaluations (optional) = surface evaluations spent, the measure
 * of what exact skipping saves.  CPU tests compare t BIT FOR BIT with the oracle's literal loop.  Needs no device. */
int rt_march_candidates_host(const double* params8, const double* inverse12, const rt_ray* rays, uint64_t n, double t_min,
                             double t_max, double best, int miss_proof, double* t_out, uint8_t* hit_out, uint64_t* evaluations);

/* Host-only build of the marcher's miss proof (csrc/rt_march.cuh (3), bernstein_clear): *clear = 1 iff the Bernstein hull
 * of  p(x) = sum_k coefficients[k] x^k  over [0, length] -- undivided, or after one / two levels of de Casteljau
 * subdivision at the midpoint -- shows |p| > threshold with the sign of p(0) on the whole interval.  degree = 4 or 6.
 * A sufficient test, never a necessary one: CPU tests compare it with dense sampling (clear => really clear) and
 * measure how often it succeeds.  Needs no device. */
int rt_bernstein_clear(const double* coefficients, int degree, double length, double threshold, int* clear);

/* Host-only self-check of the conservative cull tree k_extend walks (csrc/rt_cull.cuh): builds the tree for
 * `desc` exactly like rt_scene_create and verifies, in FP64, that every group ball encloses the balls of
 * its leaves and every root ball the balls of its groups, with the slack the proof in rt_cull.cuh needs.
 * Outputs: n_roots, n_groups (padded), n_tree (shapes under the tree), n_flat (shapes tested one by one),
 * worst = the largest (member reach - node radius) / node radius found.  The node radius is read back from
 * the FP32 table entry, which costs ~1e-8 relative; the entry itself carries a 1e-4 relative margin for the
 * FP32 roundings (the factor 1.0101 instead of 1.01), so worst <= 1e-7 means every node encloses its members.
 * Needs no device. */
int rt_cull_tree_check(const rt_scene_desc* desc, uint32_t* n_roots, uint32_t* n_groups, uint32_t* n_tree,
                       uint32_t* n_flat, double* worst);

/* Host-only emulation of the cull decisions k_extend takes (same FP32 operations, each rounded once): for every
 * ray, reached[r * n_shapes + i] = 1 when shape i would be handed to its exact test -- flat-list entry passed,
 * or root, group and leaf balls all passed, or (ray-marched shape) the ball around its marching bound passed --
 * and 0 when it is skipped.  CPU tests check "the oracle's test hits shape i  =>  reached" pair by pair. */
int rt_cull_reached(const rt_scene_desc* desc, const rt_ray* rays, uint64_t n_rays, uint8_t* reached);

/* FP64 / FP32 FMA micro-benchmarks used as roofline denominators (TFLOP/s, FMA = 2 flop). */
int rt_measure_peaks(int device, double* fp64_tflops, double* fp32_tflops);

#ifdef __cplusplus
}
#endif
#endif /* RT_B200_H */
