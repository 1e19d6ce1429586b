// rt_core.cu — the CUDA core behind include/rt_b200.h (sm_100a).
//
// Kernels
//   k_intersect_batch   batched nearest hit (Scene::closest_hit with ShapeCollection semantics)
//   k_raygen            MultisamplerRayCaster::next for a batch of pixels x samples
//   k_bounce            one segment of ray_color for every live path: nearest hit, scatter / emit /
//                       sky, survivors compacted into the next queue (ballot + popc + one atomic per warp)
//   k_resolve           per-pixel mean (trace_pixel_samples) -> (f64 sums, samples) accumulator + f64 frame
//   k_load_groups       caller-supplied rays of groups of any size -> level-0 queue + RNG keys (trace_pixel_samples_group)
//   k_group_resolve     per-group mean of caller-supplied rays, continued across the batches of a large group
//   k_adaptive_select   adaptive frames: stopping rule per pixel at a pass boundary -> list of the pixels that go on
//   k_raygen_list       adaptive frames: level-0 loader of a refinement batch (listed pixels x the pass's samples)
//   k_resolve_list      adaptive frames: continue a listed pixel's rgb and luminance sums over its new samples
//   k_assemble          multi-GPU: gathered tile-packed shards -> frame
//   k_tonemap           the bins' sqrt / clamp / *256 -> RGBA8
// Compile with -fmad=false (see rt_math.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "march_bounds.hpp"
#include "rt_queues.cuh"

using namespace rt;

// ------------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
    } while (0)

// Tiles are numbered row-major with tile row ty rotated by ty * skew positions (tile number k sits at column
// (k % tiles_x + ty * skew) % tiles_x of row ty = k / tiles_x), and tile k belongs to shard k % shard_count.  The
// rotation matters when tiles_x is a multiple of the shard count -- 1024 / 32 = 32 tiles per row on 8 GPUs: without
// it every shard owns whole COLUMNS of tiles and the shards whose columns cross the expensive object finish 25 %
// after the others (measured on cornell_box); with skew = 1 the columns become diagonals.
struct ShardMap {  // which pixels this handle owns, in "owned order" (tile-major)
    uint32_t width, height, tile_w, tile_h, tiles_x, tiles_y, shard_count, shard_index, skew;
    __host__ __device__ uint32_t tile_pixels() const { return tile_w * tile_h; }
    // owned pixel index -> (x, y); false for the padding of clipped border tiles
    __host__ __device__ bool pixel_of(uint64_t q, uint32_t& x, uint32_t& y) const {
        uint32_t tp = tile_w * tile_h;
        uint32_t j, r;
        if ((q >> 32) == 0) {  // 32-bit division whenever the index allows (a 64-bit one is ~100 instructions)
            const uint32_t q32 = (uint32_t)q;
            j = q32 / tp;
            r = q32 - j * tp;
        } else {
            j = (uint32_t)(q / tp);
            r = (uint32_t)(q % tp);
        }
        uint32_t k = shard_index + j * shard_count;
        uint32_t ty = k / tiles_x, tx = (k % tiles_x + (ty % tiles_x) * skew) % tiles_x;
        x = tx * tile_w + r % tile_w;
        y = ty * tile_h + r / tile_w;
        return x < width && y < height;
    }
};

static ShardMap make_shard_map(const rt_render_params& p, uint32_t shard_index) {
    ShardMap m;
    m.width = p.image.width;
    m.height = p.image.height;
    m.shard_count = p.shard_count ? p.shard_count : 1;
    m.shard_index = shard_index;
    m.skew = m.shard_count == 1 ? 0u : 1u;
    if (m.shard_count == 1) {  // whole image: rows, so owned order == x + y*width
        m.tile_w = m.width;
        m.tile_h = 1;
    } else {
        m.tile_w = p.tile_width ? p.tile_width : 32;
        m.tile_h = p.tile_height ? p.tile_height : 32;
    }
    m.tiles_x = (uint32_t)(((uint64_t)m.width + m.tile_w - 1) / m.tile_w);
    m.tiles_y = (uint32_t)(((uint64_t)m.height + m.tile_h - 1) / m.tile_h);
    return m;
}
// tile_pixels() and the owned-order index arithmetic are 32-bit: a tile must hold fewer than 2^32 pixels
static bool tile_fits(const ShardMap& m) { return (uint64_t)m.tile_w * m.tile_h <= 0xFFFFFFFFull; }
static uint64_t owned_tiles(const ShardMap& m) {
    uint64_t total = (uint64_t)m.tiles_x * m.tiles_y;
    if (m.shard_index >= total) return 0;
    return (total - m.shard_index + m.shard_count - 1) / m.shard_count;
}

struct RayCasterDev {  // MultisamplerRayCaster, src/camera/ray_caster.rs:17-48
    D3 camera_position, camera_right, camera_up, left_top;
    double pixel_resolution;
};

// ------------------------------------------------------------------------------------------------
// shared-memory staging of the cull tree (rt_cull.cuh; 16 B per root / group / leaf / flat entry): the
// flat list, the roots and the groups are read by every lane at the same address (broadcast), the leaves
// of a lane's own groups at per-lane addresses.  The FP64 inverse rows are only needed for the few
// survivors of the cull and stay in global memory / L1.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ Staged stage_scene(const DevScene& S, bool use_smem) {
    if (!use_smem) return Staged{false};
    float4* s_tab = reinterpret_cast<float4*>(rt_smem_raw);
    const int n = S.ctab_entries();
    for (int k = threadIdx.x; k < n; k += blockDim.x) s_tab[k] = S.ctab[k];
    // the flat list's shape records (rt_scene.cuh, FlatRec) behind the table, 16 B at a time
    const float4* frec = reinterpret_cast<const float4*>(S.frec);
    const int nf = S.n_frec * (RT_FLAT_REC * 8 / 16);
    for (int k = threadIdx.x; k < nf; k += blockDim.x) s_tab[n + k] = frec[k];
    __syncthreads();
    return Staged{true};
}

// ------------------------------------------------------------------------------------------------
// K2/K3: batched nearest hit
// ------------------------------------------------------------------------------------------------
// RT_ISECT_VERIFY support: every analytic (ray, shape) pair the cull rejects -- at its root, its group or
// its own leaf entry -- is tested exactly with max_t = +inf; a hit (or a degenerate branch) there is a
// false cull.
__device__ __noinline__ unsigned long long count_false_culls(const DevScene& S, D3 ro, D3 rd, double min_t) {
    const CullRay cr = make_cull_ray(ro.x, ro.y, ro.z, rd.x, rd.y, rd.z);
    unsigned long long bad = 0;
    for (int k = 0; k < S.n_march; k++) {  // a culled marching bound must be a miss of intersect_bound
        if (cull_pass(cr, S.march_cull[k])) continue;
        const int i = S.march_index[k];
        double start, end;
        if (march_bound(S.params + RT_SHAPE_PARAMS * i, xf_point(S.inv + 12 * i, ro), xf_vector(S.inv + 12 * i, rd), start, end)) bad++;
    }
    for (int i = 0; i < S.n_shapes; i++) {
        const int g = S.cull_group[i];
        if (g == -2) continue;
        bool reached = cull_pass(cr, S.cull[i]);
        if (g >= 0)
            reached = reached && cull_pass_node(cr, S.ctab[g / RT_CULL_ROOT_FANOUT]) && cull_pass_node(cr, S.ctab[S.n_roots + g]);
        if (g >= 0)
            for (int l = 1; l <= S.n_upper; l++)   // every ancestor above the root
                reached = reached && cull_pass_node(cr, S.cupper[S.upper_off[l] + ((g / RT_CULL_ROOT_FANOUT) >> (5 * l))]);
        if (reached) continue;
        double best = INFINITY;
        int winner = -1;
        bool degenerate = false;
        DevCounters cc = {};
        if (S.kind[i] == RT_SHAPE_TORUS) {   // (analytic_test only marks a reached torus for the replay: test it exactly here)
            double t;
            if (shape_candidate<false>(S, i, RT_SHAPE_TORUS, S.inv + 12 * i, ro, rd, min_t, INFINITY, t, cc)) bad++;
            continue;
        }
        analytic_test<false>(S, i, ro, rd, min_t, best, winner, degenerate, cc);
        if (winner >= 0 || degenerate) bad++;
    }
    return bad;
}

// MODE: RT_ISECT_BRUTE / RT_ISECT_FAST / RT_ISECT_VERIFY
template <bool COUNT, int MODE>
__global__ void __launch_bounds__(256)
k_intersect_batch(DevScene S, bool use_smem, const rt_ray* __restrict__ rays, unsigned long long n, double t_min,
                  double t_max, int32_t* __restrict__ shape_index, double* __restrict__ t_out,
                  rt_vec3* __restrict__ normal, rt_vec3* __restrict__ point, double* __restrict__ uv,
                  uint8_t* __restrict__ front_face, DevCounters* g_counters) {
    Staged st = stage_scene(S, use_smem);
    DevCounters c = {};
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        rt_ray r = rays[i];
        D3 ro = mk(r.origin.x, r.origin.y, r.origin.z), rd = mk(r.direction.x, r.direction.y, r.direction.z);
        double bt;
        int bi;
        if (MODE == RT_ISECT_BRUTE) {
            nearest_hit_brute<COUNT>(S, ro, rd, t_min, t_max, bt, bi, c);
        } else if (MODE == RT_ISECT_FAST) {
            nearest_hit_fast<COUNT>(S, st, ro, rd, t_min, t_max, bt, bi, c);
        } else {
            double ft;
            int fi;
            DevCounters cc = {};
            nearest_hit_fast<false>(S, st, ro, rd, t_min, t_max, ft, fi, cc);
            nearest_hit_brute<COUNT>(S, ro, rd, t_min, t_max, bt, bi, c);
            if (fi != bi || (bi >= 0 && __double_as_longlong(ft) != __double_as_longlong(bt))) c.verify_rays++;
            c.verify_false_culls += count_false_culls(S, ro, rd, t_min);
        }
        if (shape_index) shape_index[i] = bi;
        if (bi < 0) {
            if (t_out) t_out[i] = 0.0;
            if (normal) normal[i] = rt_vec3{0.0, 0.0, 0.0};
            if (point) point[i] = rt_vec3{0.0, 0.0, 0.0};
            if (uv) { uv[2 * i] = 0.0; uv[2 * i + 1] = 0.0; }
            if (front_face) front_face[i] = 0;
            continue;
        }
        if (t_out) t_out[i] = bt;
        if (normal || point || uv || front_face) {
            HitRec h;
            finalize_hit(S, bi, bt, ro, rd, h);
            if (normal) normal[i] = rt_vec3{h.normal.x, h.normal.y, h.normal.z};
            if (point) point[i] = rt_vec3{h.point.x, h.point.y, h.point.z};
            if (uv) { uv[2 * i] = h.u; uv[2 * i + 1] = h.v; }
            if (front_face) front_face[i] = h.front ? 1 : 0;
        }
    }
    if (COUNT || MODE == RT_ISECT_VERIFY) flush_counters(c, g_counters);
}

// ------------------------------------------------------------------------------------------------
// wavefront path tracer
// ------------------------------------------------------------------------------------------------
// warp-aggregated append: returns this lane's slot in the destination queue (valid when `alive`)

// K1: primary rays.  Batch = pixels [first_owned, first_owned + n_pixels) of this shard x spp samples,
// path id = pixel_local * spp + sample.  Padding pixels of clipped tiles produce no path.
__global__ void __launch_bounds__(256)
k_raygen(RayCasterDev rc, ShardMap map, unsigned long long first_owned, uint32_t n_pixels, uint32_t spp,
         uint32_t k0, uint32_t k1, PathQueue q, uint32_t* count_out, float4* __restrict__ radiance,
         uint2* __restrict__ path_key, uint32_t sample_base) {
    const unsigned long long n = (unsigned long long)n_pixels * spp;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    // round the trip count up so that whole warps stay converged for the ballot in queue_append
    const unsigned long long n_round = (n + 31ull) & ~31ull;
    for (unsigned long long id = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; id < n_round; id += stride) {
        bool alive = false;
        D3 dir = mk(0.0, 0.0, 0.0);
        if (id < n) {
            // (a batch holds fewer than 2^32 paths -- rt_render_start checks -- so the division is a 32-bit one)
            const uint32_t id32 = (uint32_t)id;
            uint32_t pl = id32 / spp, s = id32 - pl * spp;
            uint32_t x, y;
            if (map.pixel_of(first_owned + pl, x, y)) {
                PathRng rng;
                rng.k0 = k0; rng.k1 = k1;
                rng.pixel = x + y * map.width;
                rng.sample = sample_base + s;  // (samples of earlier frames of a progressive accumulation come first)
                rng.begin_event(0);
                double u = rng.next();   // ray_caster.rs:106-107
                double v = rng.next();
                // :109-112
                D3 d = rc.left_top + (rc.pixel_resolution * ((double)x + u)) * rc.camera_right -
                       (rc.pixel_resolution * ((double)y + v)) * rc.camera_up;
                dir = normalize(d - rc.camera_position);  // Ray::new
                path_key[id] = make_uint2(rng.pixel, rng.sample);
                alive = true;
            } else {
                radiance[id] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        uint32_t slot = queue_append(alive, count_out);
        if (alive) {
            q.ox[slot] = rc.camera_position.x; q.oy[slot] = rc.camera_position.y; q.oz[slot] = rc.camera_position.z;
            q.dx[slot] = dir.x; q.dy[slot] = dir.y; q.dz[slot] = dir.z;
            q.bx[slot] = 1.0; q.by[slot] = 1.0; q.bz[slot] = 1.0;
            q.pid[slot] = (uint32_t)id;
        }
    }
}

// One segment of ray_color (src/renderer/mod.rs:23-45), iteratively: `level` = number of hits so
// far, the reference's `depth` argument at this call is max_depth - level.
template <bool COUNT>
__global__ void __launch_bounds__(256)
k_bounce(DevScene S, bool use_smem, PathQueue in, const uint32_t* __restrict__ count_in, PathQueue out,
         uint32_t* count_out, uint32_t level, uint32_t max_depth, const uint2* __restrict__ path_key, uint32_t k0,
         uint32_t k1, float4* __restrict__ radiance, DevCounters* g_counters) {
    Staged st = stage_scene(S, use_smem);
    DevCounters c = {};
    const uint32_t n = *count_in;
    const uint32_t n_round = (n + 31u) & ~31u;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
        bool alive = false;
        D3 no = mk(0, 0, 0), nd = mk(0, 0, 0), nb = mk(0, 0, 0);
        uint32_t pid = 0;
        if (i < n) {
            D3 ro = mk(in.ox[i], in.oy[i], in.oz[i]);
            D3 rd = mk(in.dx[i], in.dy[i], in.dz[i]);
            D3 beta = mk(in.bx[i], in.by[i], in.bz[i]);
            pid = in.pid[i];
            double bt;
            int bi;
            nearest_hit_fast<COUNT>(S, st, ro, rd, 0.001, INFINITY, bt, bi, c);  // mod.rs:24
            D3 L = mk(0.0, 0.0, 0.0);
            if (bi < 0) {
                L = hadamard(beta, sky(rd));  // :41-43
            } else if (level == max_depth) {
                // depth == 0: black (:26-27)
            } else {
                HitRec h;
                finalize_hit(S, bi, bt, ro, rd, h);
                const uint2 key = path_key[pid];   // written by k_raygen / k_load_groups, as k_shade reads it
                PathRng rng;
                rng.k0 = k0; rng.k1 = k1;
                rng.pixel = key.x;
                rng.sample = key.y;
                rng.begin_event(level + 1);
                D3 ndir, atten;
                if (scatter_or_emit(S, h, rd, rng, ndir, atten)) {  // :29-32
                    alive = true;
                    no = h.point;
                    nd = ndir;
                    nb = hadamard(beta, atten);
                } else {
                    L = hadamard(beta, atten);  // :34-36
                }
            }
            if (!alive) radiance[pid] = make_float4((float)L.x, (float)L.y, (float)L.z, 1.0f);
        }
        uint32_t slot = queue_append(alive, count_out);
        if (alive) {
            out.ox[slot] = no.x; out.oy[slot] = no.y; out.oz[slot] = no.z;
            out.dx[slot] = nd.x; out.dy[slot] = nd.y; out.dz[slot] = nd.z;
            out.bx[slot] = nb.x; out.by[slot] = nb.y; out.bz[slot] = nb.z;
            out.pid[slot] = pid;
        }
    }
    if (COUNT) flush_counters(c, g_counters);
}

// ---- the wavefront proper: extend -> march -> shade ---------------------------------------------
// Splitting the segment into three kernels keeps the expensive, rare and irregular part — marching an
// implicit surface — out of the regular one: k_extend runs the analytic shape list with every lane
// busy and only QUEUES the rays whose bounding chord can still beat their best analytic hit; k_march
// runs those rays densely packed; k_shade finalises the winner, scatters and compacts the survivors.

// The primary ray of sample `sample` of pixel (x, y): MultisamplerRayCaster::next, src/camera/ray_caster.rs:100-118 --
// the two draws of event 0 of the path's RNG, then the jittered viewport point and Ray::new.  The one place this
// arithmetic lives: k_extend's raygen and k_raygen_list (adaptive refinement passes) both call it.
__device__ __forceinline__ D3 camera_ray_dir(const RayCasterDev& rc, uint32_t x, uint32_t y, uint32_t pixel,
                                            uint32_t sample, uint32_t k0, uint32_t k1) {
    PathRng rng;
    rng.k0 = k0; rng.k1 = k1;
    rng.pixel = pixel;
    rng.sample = sample;
    rng.begin_event(0);
    const double u = rng.next();   // ray_caster.rs:106-107
    const double v = rng.next();
    // :109-112
    const D3 d = rc.left_top + (rc.pixel_resolution * ((double)x + u)) * rc.camera_right -
                 (rc.pixel_resolution * ((double)y + v)) * rc.camera_up;
    return normalize(d - rc.camera_position);  // Ray::new
}

#ifndef RT_EXTEND_MIN_BLOCKS
#define RT_EXTEND_MIN_BLOCKS 3
#endif
// RAYGEN (bounce level 0 of a frame): the primary rays are GENERATED here instead of being read back from the
// queue a separate k_raygen pass wrote (that pass was a pure HBM round trip: 76 B written and 48 B re-read per path,
// 3 % of the step) -- MultisamplerRayCaster::next, src/camera/ray_caster.rs:100-118, same draws, same arithmetic.
// Path i of the batch takes queue slot i (no compaction); the slots of a clipped border tile's padding pixels
// become misses with zero throughput.
struct RaygenArgs {
    RayCasterDev rc;
    ShardMap map;
    unsigned long long first_owned;
    uint32_t n_paths, spp, k0, k1, sample_base;
    float4* radiance;
    uint32_t* count_out;   // receives n_paths: the live count of level 0 that k_march / k_shade read
};
template <bool COUNT, bool RAYGEN>
__global__ void __launch_bounds__(256, RT_EXTEND_MIN_BLOCKS)
k_extend(DevScene S, bool use_smem, PathQueue in, const uint32_t* __restrict__ count_in, HitQueue hq,
         uint32_t* march_count, uint32_t* replay_count, DevCounters* g_counters, bool any_hit_suffices,
         bool defer_bound, RaygenArgs rg) {
    Staged st = stage_scene(S, use_smem);
    DevCounters c = {};
    const uint32_t n = RAYGEN ? rg.n_paths : *count_in;
    if (RAYGEN && blockIdx.x == 0 && threadIdx.x == 0) *rg.count_out = n;
    const uint32_t n_round = (n + 31u) & ~31u;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
        uint32_t mask = 0;
        bool degenerate = false;
        bool live = i < n;
        D3 ro = mk(0.0, 0.0, 0.0), rd = mk(0.0, 0.0, 0.0);
        if (RAYGEN && live) {
            const uint32_t pl = i / rg.spp, s = i - pl * rg.spp;
            uint32_t x, y;
            if (rg.map.pixel_of(rg.first_owned + pl, x, y)) {
                const uint32_t pixel = x + y * rg.map.width;
                const uint32_t sample = rg.sample_base + s;  // (samples of earlier frames of a progressive accumulation come first)
                ro = rg.rc.camera_position;
                rd = camera_ray_dir(rg.rc, x, y, pixel, sample, rg.k0, rg.k1);
                hq.key[i] = make_uint2(pixel, sample);
                in.ox[i] = ro.x; in.oy[i] = ro.y; in.oz[i] = ro.z;
                in.dx[i] = rd.x; in.dy[i] = rd.y; in.dz[i] = rd.z;
                in.bx[i] = 1.0; in.by[i] = 1.0; in.bz[i] = 1.0;
                in.pid[i] = i;
            } else {
                // padding pixel of a clipped border tile: no path.  Its slot becomes a miss with zero throughput, so
                // that k_shade needs no special case (it writes radiance 0; nobody reads a padding pixel's sum)
                in.dx[i] = 0.0; in.dy[i] = 1.0; in.dz[i] = 0.0;
                in.bx[i] = 0.0; in.by[i] = 0.0; in.bz[i] = 0.0;
                in.pid[i] = i;
                hq.index[i] = -1;
                live = false;
            }
        }
        if (live) {
            if (!RAYGEN) {
                ro = mk(in.ox[i], in.oy[i], in.oz[i]);
                rd = mk(in.dx[i], in.dy[i], in.dz[i]);
            }
            double best;
            int winner;
            const CullRay cr = make_cull_ray(ro.x, ro.y, ro.z, rd.x, rd.y, rd.z);
            degenerate = analytic_nearest<COUNT>(S, st, cr, ro, rd, 0.001, INFINITY, best, winner, c);
            // depth == 0 (renderer/mod.rs:26-27): a hit is black whatever it is, so a ray that already hit an
            // analytic shape needs no marching at the last level
            if (!degenerate && !(any_hit_suffices && winner >= 0)) {
                for (int k = 0; k < S.n_march; k++) {
                    if (!cull_pass(cr, S.march_cull[k])) continue;  // the line misses the marching bound
                    if (defer_bound) {  // k_march_filter runs march_needed, with full warps
                        mask |= 1u << k;
                        continue;
                    }
                    const int si = S.march_index[k];
                    D3 o, d;
                    double start, end_c;
                    if (march_needed(S, S.inv + 12 * si, S.params + RT_SHAPE_PARAMS * si, ro, rd, best, o, d, start, end_c))
                        mask |= 1u << k;
                }
                if (COUNT) c.cull_tests += S.n_march;
            }
            if (COUNT) c.segments++;
            hq.t[i] = best;
            hq.index[i] = winner;
        }
        uint32_t slot = queue_append(mask != 0, march_count);
        if (mask != 0) {
            hq.mq_slot[slot] = i;
            hq.mq_mask[slot] = mask;
        }
        slot = queue_append(degenerate, replay_count);
        if (degenerate) hq.rq_slot[slot] = i;
    }
    if (COUNT) flush_counters(c, g_counters);
}

// degenerate rays: the literal ShapeCollection loop, in index order (SURVEY A.3)
__global__ void __launch_bounds__(128)
k_replay(DevScene S, PathQueue in, HitQueue hq, const uint32_t* __restrict__ replay_count) {
    const uint32_t n = *replay_count;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        const uint32_t i = hq.rq_slot[j];
        D3 ro = mk(in.ox[i], in.oy[i], in.oz[i]);
        D3 rd = mk(in.dx[i], in.dy[i], in.dz[i]);
        double best;
        int winner;
        DevCounters cc = {};
        nearest_hit_brute<false>(S, ro, rd, 0.001, INFINITY, best, winner, cc);
        hq.t[i] = best;
        hq.index[i] = winner;
    }
}

// One path segment's shade step: slot i of the input queue when `valid` (all 32 lanes of a warp call this together:
// the unit-ball sample is drawn warp-cooperatively and the survivors are appended with one atomic per warp).
__device__ __forceinline__ void shade_slot(const DevScene& S, const PathQueue& in, const HitQueue& hq, const PathQueue& out,
                                           uint32_t* count_out, uint32_t level, uint32_t max_depth, uint32_t k0, uint32_t k1,
                                           float4* __restrict__ radiance, uint4* s_id, uint32_t i, bool valid) {
    bool alive = false, shading = false, need_ball = false;
    D3 no = mk(0, 0, 0), nd = mk(0, 0, 0), nb = mk(0, 0, 0);
    D3 rd = mk(0, 0, 0), beta = mk(0, 0, 0), L = mk(0.0, 0.0, 0.0);
    uint32_t pid = 0;
    HitRec h;
    PathRng rng;
    rng.k0 = k0; rng.k1 = k1;
    rng.pixel = 0; rng.sample = 0;
    rng.begin_event(level + 1);
    if (valid) {
        rd = mk(in.dx[i], in.dy[i], in.dz[i]);
        beta = mk(in.bx[i], in.by[i], in.bz[i]);
        pid = in.pid[i];
        const int bi = hq.index[i];
        if (bi < 0) {
            L = hadamard(beta, sky(rd));  // renderer/mod.rs:41-43
        } else if (level == max_depth) {
            // depth == 0: black (:26-27)
        } else {
            D3 ro = mk(in.ox[i], in.oy[i], in.oz[i]);
            const rt_material mat = S.materials[S.material[bi]];
            finalize_hit(S, bi, hq.t[i], ro, rd, h, material_reads_uv(S, mat));
            const uint2 key = hq.key[pid];
            rng.pixel = key.x;
            rng.sample = key.y;
            shading = true;
            need_ball = material_needs_ball(mat);
        }
    }
    const D3 ball = coop_random_in_unit_sphere(need_ball, rng.pixel, rng.sample, level + 1, k0, k1, s_id);
    if (shading) {
        D3 ndir, atten;
        if (scatter_or_emit(S, h, rd, rng, ndir, atten, &ball)) {  // :29-32
            alive = true;
            no = h.point;
            nd = ndir;
            nb = hadamard(beta, atten);
        } else {
            L = hadamard(beta, atten);  // :34-36
        }
    }
    if (valid && !alive) radiance[pid] = make_float4((float)L.x, (float)L.y, (float)L.z, 1.0f);
    uint32_t slot = queue_append(alive, count_out);
    if (alive) {
        out.ox[slot] = no.x; out.oy[slot] = no.y; out.oz[slot] = no.z;
        out.dx[slot] = nd.x; out.dy[slot] = nd.y; out.dz[slot] = nd.z;
        out.bx[slot] = nb.x; out.by[slot] = nb.y; out.bz[slot] = nb.z;
        out.pid[slot] = pid;
    }
}

// K4.  BINNED = the SHADE QUEUE KEYED BY MATERIAL AND TEXTURE: the reference's 5-way Material dispatch
// (src/world/material.rs:22-31) times the nested Texture::value (src/world/texture.rs:5-8) is the divergence source of
// this kernel -- in arrival order a warp of a scene with many material kinds executes the union of their branches.
// A block therefore takes RT_SHADE_CHUNK consecutive slots, bins them in shared memory by the winner's shade key
// (0 = miss -> sky; 1 + S.mat_bin[material]: one bin per (material kind, root texture kind) pair present in the scene;
// slots past the queue's end dropped) -- a counting sort with BLOCK-AGGREGATED counters: lanes with the same key are matched inside
// the warp (__match_any_sync) and one shared-memory atomic per (warp, key) reserves their places -- and shades the
// slots in binned order, so that all but the few warps at a bin boundary run one branch.  The paths' results do not
// depend on the order (every random draw is keyed by the path), so the frame is bit-identical to the unbinned one.
// (64 registers / 4 CTAs per SM was measured: spills, 1.44 -> 1.64 ms per 4 Mi paths)
#define RT_SHADE_CHUNK 1024
#define RT_SHADE_MAX_BINS 32
// 3 CTAs per SM (<= 85 registers: the kernel needed 80 before it grew the dead-slot and binning paths; at 102 it fell
// to 2 CTAs per SM and lost 20 %)
template <bool COUNT, bool BINNED>
__global__ void __launch_bounds__(256, 3)
k_shade(DevScene S, PathQueue in, const uint32_t* __restrict__ count_in, HitQueue hq, PathQueue out, uint32_t* count_out,
        uint32_t level, uint32_t max_depth, ShardMap map, unsigned long long first_owned, uint32_t spp, uint32_t k0,
        uint32_t k1, float4* __restrict__ radiance) {
    // (map / first_owned / spp are not read -- the RNG key comes from hq.key -- but stay in the signature: dropping them
    // moves the other parameters in the constant bank and changes the generated code; measured -0.8 % on the frame)
    const uint32_t n = *count_in;
    // random_in_unit_sphere is drawn by the whole warp for its rejected lanes (coop_random_in_unit_sphere)
    __shared__ uint4 s_ball_id[256];
    uint4* const s_id = s_ball_id + (threadIdx.x & ~31u);
    if (!BINNED) {
        const uint32_t n_round = (n + 31u) & ~31u;
        const uint32_t stride = gridDim.x * blockDim.x;
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride)
            shade_slot(S, in, hq, out, count_out, level, max_depth, k0, k1, radiance, s_id, i, i < n);
        return;
    }
    __shared__ uint16_t s_order[RT_SHADE_CHUNK];
    __shared__ uint32_t s_count[RT_SHADE_MAX_BINS + 1], s_cursor[RT_SHADE_MAX_BINS + 1];
    __shared__ uint32_t s_total;
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    for (uint32_t chunk0 = blockIdx.x * RT_SHADE_CHUNK; chunk0 < n; chunk0 += gridDim.x * RT_SHADE_CHUNK) {
        if (threadIdx.x <= RT_SHADE_MAX_BINS) s_count[threadIdx.x] = 0;
        __syncthreads();
        // ---- keys + histogram: one shared atomic per (warp, key) -------------------------------------------
        int key[RT_SHADE_CHUNK / 256];
#pragma unroll
        for (int r = 0; r < RT_SHADE_CHUNK / 256; r++) {
            const uint32_t i = chunk0 + r * 256 + threadIdx.x;
            int k = -1;
            if (i < n) {
                const int bi = hq.index[i];
                k = bi < 0 ? 0 : 1 + (int)S.mat_bin[S.material[bi]];
            }
            key[r] = k;
            const unsigned peers = __match_any_sync(FULL, k);
            if (k >= 0 && lane == __ffs(peers) - 1) atomicAdd(&s_count[k], (uint32_t)__popc(peers));
        }
        __syncthreads();
        if (threadIdx.x == 0) {   // exclusive scan over at most 33 bins
            uint32_t run = 0;
            for (int k = 0; k <= RT_SHADE_MAX_BINS; k++) {
                s_cursor[k] = run;
                run += s_count[k];
            }
            s_total = run;
        }
        __syncthreads();
        // ---- places: the same matching, the warp's leader of each key reserves a run in its bin ---------------
#pragma unroll
        for (int r = 0; r < RT_SHADE_CHUNK / 256; r++) {
            const int k = key[r];
            const unsigned peers = __match_any_sync(FULL, k);
            const int leader = __ffs(peers) - 1;
            uint32_t base = 0;
            if (k >= 0 && lane == leader) base = atomicAdd(&s_cursor[k], (uint32_t)__popc(peers));
            base = __shfl_sync(FULL, base, leader);
            if (k >= 0) s_order[base + __popc(peers & ((1u << lane) - 1u))] = (uint16_t)(r * 256 + threadIdx.x);
        }
        __syncthreads();
        // ---- shade in binned order -------------------------------------------------------------------------------
        const uint32_t total = s_total, total_round = (total + 31u) & ~31u;
        for (uint32_t j = threadIdx.x; j < total_round; j += 256) {
            const bool valid = j < total;
            const uint32_t i = chunk0 + (valid ? (uint32_t)s_order[j] : 0u);
            shade_slot(S, in, hq, out, count_out, level, max_depth, k0, k1, radiance, s_id, i, valid);
        }
        __syncthreads();
    }
}

// K5: per-pixel mean of the batch (trace_pixel_samples, src/renderer/mod.rs:151-155).  One thread
// per owned pixel; the accumulator keeps (sum rgb, samples) as four doubles for the multi-GPU exchange and the
// progressive accumulation -- the f64 sums themselves, so that an assembled or accumulated frame is the very
// mean the unsharded single frame holds -- the frame buffer the f64 mean for the host path.
struct __align__(16) Acc {
    double r, g, b, n;
};
// Adaptive frames (rt_render_start_adaptive) also keep, per pixel, the f64 sums of the samples' luminance and of its
// square, in sample order: y = (0.2126 r + 0.7152 g) + 0.0722 b of the float radiance widened to double (this file is
// compiled with -fmad=false, so no product is fused into the sums).
__device__ __forceinline__ double luminance(float4 v) {
    return (0.2126 * (double)v.x + 0.7152 * (double)v.y) + 0.0722 * (double)v.z;
}
// MOMENTS: also Σy, Σy² into moments[] (pass 0 of an adaptive frame); the plain instantiation is the frame path's
template <bool MOMENTS>
__global__ void __launch_bounds__(256)
k_resolve(const float4* __restrict__ radiance, uint32_t n_pixels, uint32_t spp, unsigned long long first_owned,
          Acc* __restrict__ accum, rt_vec3* __restrict__ frame_owned, bool add, double2* __restrict__ moments) {
    uint32_t pl = blockIdx.x * blockDim.x + threadIdx.x;
    if (pl >= n_pixels) return;
    const float4* r = radiance + (size_t)pl * spp;
    double sx = 0.0, sy = 0.0, sz = 0.0, ln = (double)spp;
    double my = 0.0, myy = 0.0;
    if (add) {  // progressive accumulation: continue the earlier frames' sums, sample by sample (k frames of n
                // samples then hold the very sum one frame of k*n samples computes)
        const Acc prev = accum[first_owned + pl];
        sx = prev.r; sy = prev.g; sz = prev.b;
        ln += prev.n;
        if (MOMENTS) {
            const double2 pm = moments[first_owned + pl];
            my = pm.x; myy = pm.y;
        }
    }
    for (uint32_t s = 0; s < spp; s++) {
        float4 v = r[s];
        sx += (double)v.x; sy += (double)v.y; sz += (double)v.z;
        if (MOMENTS) {
            const double y = luminance(v);
            my += y; myy += y * y;
        }
    }
    accum[first_owned + pl] = Acc{sx, sy, sz, ln};
    frame_owned[first_owned + pl] = rt_vec3{sx / ln, sy / ln, sz / ln};
    if (MOMENTS) moments[first_owned + pl] = make_double2(my, myy);
}

// ---- adaptive sampling (rt_render_start_adaptive) -------------------------------------------------------------------
// The stopping rule, in the operation order the header documents (so that numpy can replay it bit for bit).
__device__ __forceinline__ bool adaptive_converged(double n, double sum_y, double sum_yy, double rel_error, double abs_error) {
    const double mean = sum_y / n;
    const double var = fmax(0.0, (sum_yy - sum_y * mean) / (n - 1.0));
    const double se = sqrt(var / n);
    return se <= fmax(rel_error * fabs(mean), abs_error);
}

// One thread per owned pixel: the pixels that hold n_k samples (the ones traced in the previous pass) are tested; the
// unconverged ones (while n_k < samples_number, which the host guarantees by not planning a pass past it) are appended
// to list[] -- in no particular order: every later step of a pixel depends only on its own sums -- and counted in
// *live.
__global__ void __launch_bounds__(256)
k_adaptive_select(const Acc* __restrict__ accum, const double2* __restrict__ moments, uint32_t n_pixels, double n_k,
                  double rel_error, double abs_error, uint32_t* __restrict__ list, uint32_t* live) {
    const uint32_t n_round = (n_pixels + 31u) & ~31u;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t p = blockIdx.x * blockDim.x + threadIdx.x; p < n_round; p += stride) {
        bool go = false;
        if (p < n_pixels && accum[p].n == n_k) {
            const double2 m = moments[p];
            go = !adaptive_converged(n_k, m.x, m.y, rel_error, abs_error);
        }
        const uint32_t slot = queue_append(go, live);
        if (go) list[slot] = p;
    }
}

// Level 0 of batch j of a refinement pass (modelled on k_load_groups): pixels list[base .. base + B) of the *live
// listed ones, m samples each, numbered n_k .. n_k + m - 1.  Path i takes pixel list[base + i / m] and sample
// n_k + i % m; the primary ray is the frame's own (camera_ray_dir).  *count_out = the batch's path count, 0 for a
// batch past the end of the list (every kernel of the batch then exits at once).
__global__ void __launch_bounds__(256)
k_raygen_list(RayCasterDev rc, uint32_t width, const uint32_t* __restrict__ list, const uint32_t* __restrict__ live,
              uint32_t base, uint32_t B, uint32_t m, uint32_t n_k, uint32_t k0, uint32_t k1, PathQueue q,
              uint2* __restrict__ path_key, uint32_t* count_out) {
    const uint32_t count = *live;
    const uint32_t n = count > base ? min(count - base, B) * m : 0u;   // (B * m fits in 32 bits: planned so)
    if (blockIdx.x == 0 && threadIdx.x == 0) *count_out = n;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t pl = i / m, s = i - pl * m;
        const uint32_t pixel = list[base + pl];
        const uint32_t y = pixel / width, x = pixel - y * width;
        const uint32_t sample = n_k + s;
        const D3 rd = camera_ray_dir(rc, x, y, pixel, sample, k0, k1);
        q.ox[i] = rc.camera_position.x; q.oy[i] = rc.camera_position.y; q.oz[i] = rc.camera_position.z;
        q.dx[i] = rd.x; q.dy[i] = rd.y; q.dz[i] = rd.z;
        q.bx[i] = 1.0; q.by[i] = 1.0; q.bz[i] = 1.0;
        q.pid[i] = i;
        path_key[i] = make_uint2(pixel, sample);
    }
}

// One thread per listed pixel of the batch: continue its (Σrgb, n) and (Σy, Σy²) sample by sample over its m
// contiguous radiance slots -- the very sums one frame of n + m samples computes -- and write the accumulator, the
// moments and the frame.  The loads of 16 samples are issued together, as in k_group_resolve.
__global__ void __launch_bounds__(256)
k_resolve_list(const float4* __restrict__ radiance, const uint32_t* __restrict__ list, const uint32_t* __restrict__ live,
               uint32_t base, uint32_t B, uint32_t m, Acc* __restrict__ accum, double2* __restrict__ moments,
               rt_vec3* __restrict__ frame) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t count = *live;
    if (t >= B || count <= base || t >= count - base) return;
    const uint32_t p = list[base + t];
    const Acc prev = accum[p];
    const double2 pm = moments[p];
    double sx = prev.r, sy = prev.g, sz = prev.b, my = pm.x, myy = pm.y;
    const float4* r = radiance + (size_t)t * m;
    uint32_t s = 0;
    for (; s + 16 <= m; s += 16) {
        float4 v[16];
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = r[s + j];
#pragma unroll
        for (int j = 0; j < 16; j++) {
            sx += (double)v[j].x; sy += (double)v[j].y; sz += (double)v[j].z;
            const double y = luminance(v[j]);
            my += y; myy += y * y;
        }
    }
    for (; s < m; s++) {
        const float4 v = r[s];
        sx += (double)v.x; sy += (double)v.y; sz += (double)v.z;
        const double y = luminance(v);
        my += y; myy += y * y;
    }
    const double ln = prev.n + (double)m;
    accum[p] = Acc{sx, sy, sz, ln};
    moments[p] = make_double2(my, myy);
    frame[p] = rt_vec3{sx / ln, sy / ln, sz / ln};
}

// rt_render_pixel_stats: the samples each pixel holds
__global__ void __launch_bounds__(256)
k_pixel_counts(const Acc* __restrict__ accum, uint32_t n_pixels, uint32_t* __restrict__ counts) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_pixels) counts[p] = (uint32_t)accum[p].n;
}

// K5b: per-group mean of caller rays (trace_pixel_samples, src/renderer/mod.rs:151-155, per group of :127-149), one
// thread per group of the batch (rays [r0, r1), group slice as in k_load_groups).  The same arithmetic as k_resolve:
// f64 sums in sample order from 0.0, then one division by the group's ray count -- an empty group gives 0 / 0 = NaN,
// what the reference's Vector3d / 0.0 gives.  A group larger than a batch is traced in consecutive batches of ONE
// stream: its running f64 sum waits in means[k] between them, and the batch that holds its last ray divides.
__global__ void __launch_bounds__(256)
k_group_resolve(const float4* __restrict__ radiance, unsigned long long r0, unsigned long long r1,
                const unsigned long long* __restrict__ offsets, uint32_t n_groups, rt_vec3* __restrict__ means) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_groups) return;
    const unsigned long long first = offsets[k], end = offsets[k + 1];
    double sx = 0.0, sy = 0.0, sz = 0.0;
    if (first < r0) {   // continued from the previous batch
        const rt_vec3 prev = means[k];
        sx = prev.x; sy = prev.y; sz = prev.z;
    }
    const unsigned long long a = first > r0 ? first : r0, b = end < r1 ? end : r1;
    // the sum is serial (its order is the contract); the loads of 16 samples are issued together so that a large group
    // waits for memory once per 16 samples instead of once per sample
    unsigned long long r = a;
    for (; r + 16 <= b; r += 16) {
        float4 v[16];
#pragma unroll
        for (int j = 0; j < 16; j++) v[j] = radiance[r - r0 + j];
#pragma unroll
        for (int j = 0; j < 16; j++) {
            sx += (double)v[j].x; sy += (double)v[j].y; sz += (double)v[j].z;
        }
    }
    for (; r < b; r++) {
        const float4 v = radiance[r - r0];
        sx += (double)v.x; sy += (double)v.y; sz += (double)v.z;
    }
    if (end > r1) {
        means[k] = rt_vec3{sx, sy, sz};
        return;
    }
    const double n = (double)(end - first);
    means[k] = rt_vec3{sx / n, sy / n, sz / n};
}

// K7: de-interleave gathered shards into the frame (x + y*w, f64 linear mean)
struct ShardPtrs {
    const Acc* p[16];
};
__global__ void __launch_bounds__(256)
k_assemble(ShardPtrs shards, ShardMap map0, rt_vec3* __restrict__ frame) {
    // one-dimensional grid over x + y*w: gridDim.y (at most 65535) would cap the image height
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)map0.width * map0.height) return;
    const uint32_t y = (uint32_t)(i / map0.width), x = (uint32_t)(i - (uint64_t)y * map0.width);
    uint32_t tx = x / map0.tile_w, ty = y / map0.tile_h;
    uint32_t rot = ((ty % map0.tiles_x) * map0.skew) % map0.tiles_x;        // undo the row rotation of ShardMap
    uint32_t k = ty * map0.tiles_x + (tx + map0.tiles_x - rot) % map0.tiles_x;
    uint32_t s = k % map0.shard_count, j = k / map0.shard_count;
    size_t q = (size_t)j * map0.tile_pixels() + (size_t)(y % map0.tile_h) * map0.tile_w + (x % map0.tile_w);
    const Acc v = shards.p[s][q];
    frame[(size_t)y * map0.width + x] = rt_vec3{v.r / v.n, v.g / v.n, v.b / v.n};
}

// src/bin/main_raylib.rs:239-247
__global__ void __launch_bounds__(256)
k_tonemap(const rt_vec3* __restrict__ frame, unsigned long long n, uchar4* __restrict__ rgba) {
    unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    rt_vec3 c = frame[i];
    double r = sqrt(c.x), g = sqrt(c.y), b = sqrt(c.z);
    // f64::clamp keeps NaN, and `NaN as u8` is 0
    auto q = [](double v) -> unsigned char {
        if (isnan(v)) return 0;
        double cl = fmin(fmax(v, 0.0), 0.999);
        return (unsigned char)(cl * 256.0);
    };
    rgba[i] = make_uchar4(q(r), q(g), q(b), 255);
}

// K6: caller-supplied rays (trace_pixel_samples_group, src/renderer/mod.rs:127-149).  The batch is rays [r0, r0 + n)
// of the call; `offsets` is the batch's slice of the call's group offsets (offsets[k] = first ray of group k, global
// ray numbers, n_groups + 1 entries, offsets[0] <= r0 and offsets[n_groups] >= r0 + n).  Path i is ray r0 + i: its
// group is found by binary search, its RNG key is (pixel_index[group], ray number inside the group).
__global__ void __launch_bounds__(256)
k_load_groups(const rt_ray* __restrict__ rays, uint32_t n, unsigned long long r0, const unsigned long long* __restrict__ offsets,
              const uint32_t* __restrict__ pixel_index, uint32_t n_groups, PathQueue q, uint32_t* count_out,
              uint2* __restrict__ path_key) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *count_out = n;
    if (i >= n) return;
    const unsigned long long r = r0 + i;
    uint32_t lo = 0, hi = n_groups;   // the last group that starts at or before r (empty groups before it start there too)
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (offsets[mid] <= r) lo = mid; else hi = mid;
    }
    const rt_ray ray = rays[i];
    q.ox[i] = ray.origin.x; q.oy[i] = ray.origin.y; q.oz[i] = ray.origin.z;
    q.dx[i] = ray.direction.x; q.dy[i] = ray.direction.y; q.dz[i] = ray.direction.z;
    q.bx[i] = 1.0; q.by[i] = 1.0; q.bz[i] = 1.0;
    q.pid[i] = i;
    path_key[i] = make_uint2(pixel_index[lo], (uint32_t)(r - offsets[lo]));   // (groups have fewer than 2^32 rays)
}

// FMA micro-benchmarks: 8 independent chains per thread, FMA counted as 2 flop
template <typename T>
__global__ void __launch_bounds__(256) k_fma_peak(T* out, int iters, T a, T b) {
    T x0 = (T)threadIdx.x, x1 = x0 + (T)1, x2 = x0 + (T)2, x3 = x0 + (T)3, x4 = x0 + (T)4, x5 = x0 + (T)5,
      x6 = x0 + (T)6, x7 = x0 + (T)7;
    for (int i = 0; i < iters; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------

enum { RT_KCLASS_RAYGEN = 0, RT_KCLASS_EXTEND, RT_KCLASS_MARCH, RT_KCLASS_SHADE, RT_KCLASS_RESOLVE, RT_KCLASS_COUNT };

struct Batch {
    uint64_t first_owned;
    uint32_t n_pixels;
    cudaEvent_t done;
};

// One set of path-state buffers + the stream its kernels run on.  Batches alternate between
// RT_MAX_LANES lanes so that the tail of one batch's kernels (a few long marches, the thin deep bounce
// levels) overlaps with the other batch's kernels instead of leaving SMs idle.
#define RT_MAX_LANES 3
struct PathLane {
    cudaStream_t stream = nullptr;
    cudaEvent_t done = nullptr;
    PathQueue q[2]{};
    HitQueue hq{};
    float4* d_radiance = nullptr;
    uint32_t* d_counts = nullptr;
    void* d_march_state = nullptr;
    std::vector<void*> qallocs;
    uint64_t path_capacity = 0;
};

struct rt_scene {
    int device = 0;
    int n_sm = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    DevScene ds{};
    std::vector<void*> allocs;  // scene arrays
    bool use_smem = false;
    size_t smem_bytes = 0;
    int grid = 0;

    // instrumentation
    bool counters_on = false;
    DevCounters* d_counters = nullptr;
    uint64_t launches = 0, paths = 0;
    double last_frame_ms = 0.0, last_intersect_ms = 0.0;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    // per-kernel-class device time (rt_set_kernel_timing): event pairs around every launch of a frame,
    // resolved when the frame completes
    bool ktiming = false;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    struct Span { int cls; cudaEvent_t a, b; };
    std::vector<Span> spans;
    double ms_cls[RT_KCLASS_COUNT] = {0, 0, 0, 0, 0};
    uint64_t n_cls[RT_KCLASS_COUNT] = {0, 0, 0, 0, 0};

    // render state
    bool rendering = false, frame_complete = false;
    rt_render_params rp{};
    ShardMap map{};
    uint64_t owned_pixels = 0;   // incl. tile padding
    uint64_t path_capacity = 0;  // allocated queue capacity (paths)
    PathQueue q[2]{};
    std::vector<void*> qallocs;
    float4* d_radiance = nullptr;
    HitQueue hq{};
    uint32_t* d_counts = nullptr;  // RT_CNT_WORDS per batch (reset per batch), see RT_CNT_*
    int grid_extend = 0, grid_march = 0, grid_shade = 0;
    uint32_t kind_mask[6] = {0, 0, 0, 0, 0, 0};  // marched shapes (bits of the march-queue mask) per surface kind
    void* d_march_state = nullptr;               // k_march2: its records (rt_march_kernels.cu)
    int grid_march2 = 0, grid_march3 = 0;
    size_t smem_march3 = 0;
    bool defer_bound = true;                     // k_extend queues every ray whose line touches a marching bound's ball and leaves the bounding chord (march_needed: 8 % of its instructions at 7 of 32 lanes) to k_march_filter, which runs it with full warps (RT_B200_DEFER_BOUND=0: off; off without the filter)
    bool march_filter = true;                    // k_march_filter before the marching kernels (RT_B200_MARCH_FILTER=0: off)
    int march_version = 1;                       // 1: one ray per lane (k_march); RT_B200_MARCH=3: pool of rays per SM + per-phase queues
                                                 // (k_march3, rt_march3.cu: correct but slower, see profiles/); =2: block-local wavefront (k_march2)
    int3 march_tune = make_int3(8, 8, 8);        // k_march scheduling thresholds (RT_B200_MARCH_TUNE=a,b,c)
    int3 march_tune0 = make_int3(32, 8, 8);      // ... at bounce level 0 (RT_B200_MARCH_TUNE0=a,b,c): neighbouring entries are samples of one pixel, so a warp refills only when all of its lanes are done and its 32 rays stay (nearly) in step: k_march -3 % on cornell_box, -4 % on dupin
    int march_grid_scale = 100;                  // percent of the occupancy grid
    bool wavefront = true;         // extend/march/shade; false = fused k_bounce (more than 32 marched shapes)
    bool shade_binned = false;     // k_shade bins a block's slots by (material kind, texture kind) before shading them
    int n_shade_bins = 0;
    Acc* d_accum = nullptr;        // owned order: (sum r, g, b, samples)
    rt_vec3* d_frame = nullptr;    // owned order
    uint64_t frame_capacity = 0;
    // progressive accumulation (rt_render_set_accumulate): samples already in d_accum and the frame they belong to
    bool accumulate = false;
    uint32_t accumulated_spp = 0;
    rt_render_params accum_rp{};
    rt_camera accum_cam{};
    // the fields q, hq, d_radiance, d_counts, d_march_state, qallocs, path_capacity and `stream` above are
    // the BOUND lane's (bind_lane swaps them); lanes[0].stream is the main stream
    PathLane lanes[RT_MAX_LANES];
    int n_lanes = 3, cur_lane = 0;
    bool lanes_from_env = false;
    std::vector<Batch> batches;
    size_t delivered = 0;          // batches already copied to the caller
    cudaEvent_t ev_frame_start = nullptr, ev_frame_stop = nullptr;
    rt_vec3* host_stage = nullptr;    // sharded poll: owned-order staging, pinned
    uint64_t host_stage_cap = 0;
    // frame post-process on the device (rt_tonemap_rgba8[_device]): persistent buffers, grown on demand
    rt_vec3* d_tone_in = nullptr;
    uchar4* d_tone_out = nullptr;
    uint64_t tone_in_cap = 0, tone_out_cap = 0;
    // several devices behind one handle (rt_scene_create_multi): this is the handle of device_ids[0]; `peers` are
    // complete handles for the other devices.  A whole-frame rt_render_start shards the frame over all of them
    // by interleaved tiles, every shard's accumulator comes to this device by one peer copy, k_assemble builds
    // d_full_frame.
    std::vector<rt_scene*> peers;
    std::vector<Acc*> d_peer_acc;         // [peers.size()] staging for the peers' accumulators, on this device
    std::vector<uint64_t> peer_acc_cap;
    std::vector<cudaEvent_t> ev_peer;     // peer k's accumulator has arrived
    rt_vec3* d_full_frame = nullptr;      // x + y*w, f64 mean
    uint64_t full_frame_cap = 0;
    cudaEvent_t ev_multi_done = nullptr;
    bool multi_active = false;            // the frame in flight / last completed was rendered by all devices
    rt_render_params multi_rp{};
    // rt_trace_pixel_samples_group: the call's group offsets and pixel indices on the device, the host form's rays and
    // means (persistent buffers, grown on demand), and the events that order a call against the caller's stream
    unsigned long long* d_group_off = nullptr;
    uint32_t* d_group_pix = nullptr;
    rt_vec3* d_group_means = nullptr;
    rt_ray* d_group_rays = nullptr;
    uint64_t group_off_cap = 0, group_pix_cap = 0, group_means_cap = 0, group_rays_cap = 0;
    // host copies of the caller's offsets / pixel indices: pageable memory the library owns, so that the upload has read
    // them when cudaMemcpyAsync returns even if the caller's arrays are pinned (an upload from pinned memory is only
    // read when the stream gets there, after the caller may have reused them)
    std::vector<uint64_t> h_group_off;
    std::vector<uint32_t> h_group_pix;
    cudaEvent_t ev_group_in = nullptr, ev_group_start = nullptr, ev_group_done = nullptr;
    // adaptive sampling (rt_render_start_adaptive): whether the frame in flight / last completed is adaptive, its
    // per-pixel (Σy, Σy²), the pixel list of the current refinement pass, the listed count of every pass, the samples
    // every pass adds (pass 0: min_samples), and the event the lanes wait on after each k_adaptive_select
    bool adaptive_frame = false;
    double2* d_moments = nullptr;
    uint32_t* d_plist = nullptr;
    uint32_t* d_live = nullptr;
    uint64_t moments_cap = 0, plist_cap = 0, live_cap = 0;
    std::vector<uint32_t> adaptive_m;
    cudaEvent_t ev_adaptive_fork = nullptr;
    uint32_t* d_pix_counts = nullptr;   // rt_render_pixel_stats
    uint64_t pix_counts_cap = 0;
};

template <class T>
static int upload(rt_scene* sc, const T* src, size_t count, const T** out) {
    void* d = nullptr;
    size_t bytes = std::max<size_t>(count * sizeof(T), 16);
    CU(cudaMalloc(&d, bytes));
    sc->allocs.push_back(d);
    if (count) CU(cudaMemcpy(d, src, count * sizeof(T), cudaMemcpyHostToDevice));
    *out = (const T*)d;
    return RT_OK;
}

template <class T>
static int ensure_device_array(T*& p, uint64_t& cap, uint64_t n) {   // persistent buffer, grown on demand
    if (cap >= n) return RT_OK;
    cudaFree(p);
    p = nullptr;
    cap = 0;
    CU(cudaMalloc(&p, std::max<uint64_t>(n, 1) * sizeof(T)));
    cap = n;
    return RT_OK;
}

static size_t env_size(const char* name, size_t dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    return (size_t)strtoull(v, nullptr, 10);
}

extern "C" {

int rt_abi_version(void) { return RT_B200_ABI_VERSION; }
const char* rt_last_error(void) { return g_err.c_str(); }

int rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

static int validate_desc(const rt_scene_desc* d) {
    if (!d) return fail(RT_ERR_INVALID, "null scene description");
    if (d->n_shapes && (!d->kind || !d->flags || !d->inverse || !d->direct || !d->params || !d->material))
        return fail(RT_ERR_INVALID, "scene description: null shape array");
    if ((d->n_materials && !d->materials) || (d->n_textures && !d->textures) || (d->n_images && !d->images) ||
        (d->n_noise && !d->noise))
        return fail(RT_ERR_INVALID, "scene description: null table");
    for (uint32_t i = 0; i < d->n_shapes; i++) {
        if (d->kind[i] > RT_SHAPE_TORUS) return fail(RT_ERR_INVALID, "scene description: unknown shape kind");
        if (d->material[i] >= d->n_materials) return fail(RT_ERR_INVALID, "scene description: material index out of range");
        if (d->kind[i] == RT_SHAPE_MARCH) {
            double sk = d->params[(size_t)i * RT_SHAPE_PARAMS];
            if (!(sk >= 0 && sk <= RT_SURF_CUSHION)) return fail(RT_ERR_INVALID, "scene description: unknown surface kind");
        }
    }
    for (uint32_t i = 0; i < d->n_materials; i++) {
        const rt_material& m = d->materials[i];
        if (m.kind > RT_MAT_EMPTY) return fail(RT_ERR_INVALID, "scene description: unknown material kind");
        bool needs_tex = m.kind == RT_MAT_LAMBERTIAN || m.kind == RT_MAT_METAL || m.kind == RT_MAT_DIFFUSE_LIGHT;
        if (needs_tex && m.texture >= d->n_textures) return fail(RT_ERR_INVALID, "scene description: texture index out of range");
    }
    for (uint32_t i = 0; i < d->n_textures; i++) {
        const rt_texture& t = d->textures[i];
        if (t.kind > RT_TEX_NOISE) return fail(RT_ERR_INVALID, "scene description: unknown texture kind");
        if (t.kind == RT_TEX_NOISE && (t.image >= d->n_noise || !d->noise)) return fail(RT_ERR_INVALID, "scene description: noise index out of range");
        if ((t.kind == RT_TEX_CHECKER || t.kind == RT_TEX_UV_CHECKER) && (t.odd >= d->n_textures || t.even >= d->n_textures))
            return fail(RT_ERR_INVALID, "scene description: child texture index out of range");
        if (t.kind == RT_TEX_IMAGE && t.image >= d->n_images) return fail(RT_ERR_INVALID, "scene description: image index out of range");
    }
    {   // texture_value follows at most RT_TEX_MAX_DEPTH checker edges.  Let H(i) be the number of checker edges on the
        // longest path down from texture i (infinite on a cycle).  h[i] never exceeds H(i), and after sweep r it is at
        // least min(r, H(i)); so RT_TEX_MAX_DEPTH + 1 sweeps find every texture that is too deep or on a cycle, without
        // recursion.
        std::vector<uint8_t> h(d->n_textures, 0);
        for (int r = 0; r <= RT_TEX_MAX_DEPTH; r++)
            for (uint32_t i = 0; i < d->n_textures; i++) {
                const rt_texture& t = d->textures[i];
                if (t.kind == RT_TEX_CHECKER || t.kind == RT_TEX_UV_CHECKER)
                    h[i] = (uint8_t)std::min(1 + std::max(h[t.odd], h[t.even]), RT_TEX_MAX_DEPTH + 1);
            }
        for (uint32_t i = 0; i < d->n_textures; i++)
            if (h[i] > RT_TEX_MAX_DEPTH)
                return fail(RT_ERR_INVALID, "scene description: texture graph cyclic or deeper than RT_TEX_MAX_DEPTH");
    }
    for (uint32_t i = 0; i < d->n_noise; i++) {
        const rt_perlin& pn = d->noise[i];
        for (int k = 0; k < 256; k++)
            if (pn.perm_x[k] > 255 || pn.perm_y[k] > 255 || pn.perm_z[k] > 255)
                return fail(RT_ERR_INVALID, "scene description: Perlin permutation entry out of range");
    }
    for (uint32_t i = 0; i < d->n_images; i++) {
        if (!d->images[i].rgba || !d->images[i].width || !d->images[i].height)
            return fail(RT_ERR_INVALID, "scene description: empty image");
        if ((uint64_t)d->images[i].width * d->images[i].height > SIZE_MAX / 4)
            return fail(RT_ERR_INVALID, "scene description: image too large to address");
    }
    return RT_OK;
}

int rt_scene_create(const rt_scene_desc* d, int device, rt_scene** out) {
    if (!out) return fail(RT_ERR_INVALID, "null out pointer");
    *out = nullptr;
    int rc = validate_desc(d);
    if (rc != RT_OK) return rc;
    int ndev = rt_device_count();
    if (ndev == 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device: the path-tracing core has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(RT_ERR_INVALID, "device index out of range");
    CU(cudaSetDevice(device));
    rt_scene* sc = new rt_scene();
    sc->device = device;
    auto bail = [&](int code) {
        rt_scene_destroy(sc);
        return code;
    };
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(fail(RT_ERR_CUDA, "cudaGetDeviceProperties failed"));
    sc->n_sm = prop.multiProcessorCount;
    sc->smem_optin = prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&sc->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&sc->copy_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(RT_ERR_CUDA, "cudaStreamCreate failed"));
    sc->lanes[0].stream = sc->stream;
    for (int l = 1; l < RT_MAX_LANES; l++) {
        if (cudaStreamCreateWithFlags(&sc->lanes[l].stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&sc->lanes[l].done, cudaEventDisableTiming) != cudaSuccess)
            return bail(fail(RT_ERR_CUDA, "cudaStreamCreate failed"));
    }
    // three lanes since round 2 (the marching kernels got shorter, the thin deep levels weigh more: 944 -> 957 Mpaths/s on
    // the bench frame); a frame of fewer than 6 batches takes two of them (4 batches on 3 lanes end with a batch alone)
    sc->n_lanes = (int)std::min<size_t>(std::max<size_t>(env_size("RT_B200_LANES", 3), 1), RT_MAX_LANES);
    sc->lanes_from_env = getenv("RT_B200_LANES") != nullptr;
    cudaEventCreate(&sc->ev_a);
    cudaEventCreate(&sc->ev_b);
    cudaEventCreate(&sc->ev_frame_start);
    cudaEventCreate(&sc->ev_frame_stop);
    if (cudaEventCreateWithFlags(&sc->ev_group_in, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&sc->ev_group_start, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&sc->ev_group_done, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&sc->ev_adaptive_fork, cudaEventDisableTiming) != cudaSuccess)
        return bail(fail(RT_ERR_CUDA, "cudaEventCreate failed"));

    const uint32_t n = d->n_shapes;
    sc->ds.n_shapes = (int)n;
    if ((rc = upload(sc, d->inverse, (size_t)n * 12, &sc->ds.inv)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->direct, (size_t)n * 12, &sc->ds.dir)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->params, (size_t)n * RT_SHAPE_PARAMS, &sc->ds.params)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->kind, (size_t)n, &sc->ds.kind)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->flags, (size_t)n, &sc->ds.flags)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->material, (size_t)n, &sc->ds.material)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->materials, (size_t)d->n_materials, &sc->ds.materials)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->textures, (size_t)d->n_textures, &sc->ds.textures)) != RT_OK) return bail(rc);
    {   // shade keys: one bin per (material kind, root texture kind) pair present in the scene (k_shade, BINNED)
        std::vector<uint8_t> mat_bin(d->n_materials, 0);
        std::vector<int> seen;   // pair codes in order of first appearance
        for (uint32_t i = 0; i < d->n_materials; i++) {
            const rt_material& m = d->materials[i];
            const bool has_tex = m.kind == RT_MAT_LAMBERTIAN || m.kind == RT_MAT_METAL || m.kind == RT_MAT_DIFFUSE_LIGHT;
            int code = (int)m.kind * 16 + (has_tex ? (int)d->textures[m.texture].kind : 15);
            if (m.kind == RT_MAT_METAL && m.scalar == 0.0) code += 8;   // (a mirror draws no unit-ball sample)
            size_t b = std::find(seen.begin(), seen.end(), code) - seen.begin();
            if (b == seen.size()) seen.push_back(code);
            mat_bin[i] = (uint8_t)std::min<size_t>(b, RT_SHADE_MAX_BINS - 1);
        }
        if ((rc = upload(sc, mat_bin.data(), mat_bin.size(), &sc->ds.mat_bin)) != RT_OK) return bail(rc);
        // Binning pays when a warp in arrival order would see many keys: measured on the all-materials variant of
        // detached_materials.json (8 keys; k_shade at bounce levels 1 / 2: 15 / 13 -> 28 / 28 of 32 lanes, 332 / 142 ->
        // 188 / 83 us, frame + 8 %) against cornell_box.json (4 keys, nearly every hit Lambertian: - 0.6 %).  So: on
        // by default when the shapes of the scene reference at least 5 different keys; RT_B200_SHADE_BINNED=0 / 1 overrides.
        std::vector<char> used(seen.size(), 0);
        for (uint32_t i = 0; i < n; i++) used[std::min<size_t>(mat_bin[d->material[i]], used.size() - 1)] = 1;
        sc->n_shade_bins = (int)std::count(used.begin(), used.end(), 1);
        const char* sb = getenv("RT_B200_SHADE_BINNED");
        sc->shade_binned = sb ? atoi(sb) != 0 : sc->n_shade_bins >= 5;
    }
    std::vector<DevImage> imgs(d->n_images);
    for (uint32_t i = 0; i < d->n_images; i++) {
        imgs[i].width = d->images[i].width;
        imgs[i].height = d->images[i].height;
        if ((rc = upload(sc, d->images[i].rgba, (size_t)4 * imgs[i].width * imgs[i].height, &imgs[i].rgba)) != RT_OK) return bail(rc);
    }
    if ((rc = upload(sc, imgs.data(), imgs.size(), &sc->ds.images)) != RT_OK) return bail(rc);
    if ((rc = upload(sc, d->noise, (size_t)d->n_noise, &sc->ds.noise)) != RT_OK) return bail(rc);
    std::vector<int> march;
    for (uint32_t i = 0; i < n; i++)
        if (d->kind[i] == RT_SHAPE_MARCH) march.push_back((int)i);
    sc->ds.n_march = (int)march.size();
    if ((rc = upload(sc, march.data(), march.size(), &sc->ds.march_index)) != RT_OK) return bail(rc);
    // exact-skip marching: gradient bound of each marched surface over its region (rt_march.cuh)
    std::vector<double> march_G(march.size());
    for (size_t k = 0; k < march.size(); k++) {
        double H;
        bounds::region_bounds(d->params + (size_t)march[k] * RT_SHAPE_PARAMS, &march_G[k], &H);
        if (getenv("RT_B200_NO_MARCH_SKIP")) march_G[k] = INFINITY;
    }
    if ((rc = upload(sc, march_G.data(), march_G.size(), &sc->ds.march_G)) != RT_OK) return bail(rc);
    std::vector<double> march_F(march.size());
    for (size_t k = 0; k < march.size(); k++) {
        const double* q = d->params + (size_t)march[k] * RT_SHAPE_PARAMS;
        march_F[k] = bounds::region_magnitude(q);
        if (k < 32) sc->kind_mask[(int)q[0]] |= 1u << k;
    }
    if ((rc = upload(sc, march_F.data(), march_F.size(), &sc->ds.march_F)) != RT_OK) return bail(rc);
    std::vector<float4> march_cull(march.size());
    for (size_t k = 0; k < march.size(); k++) {
        const double* q = d->params + (size_t)march[k] * RT_SHAPE_PARAMS;
        double radius[3] = {q[7], q[7], q[7]};
        if ((int)q[0] == RT_SURF_HEART) { radius[0] = 1.45; radius[1] = 1.45 / 2.05; radius[2] = 1.45; }  // march_bound
        march_cull[k] = cull_entry_march_bound(d->inverse + (size_t)12 * march[k], radius);
        if (getenv("RT_B200_NO_CULL")) march_cull[k].w = INFINITY;
    }
    if ((rc = upload(sc, march_cull.data(), march_cull.size(), &sc->ds.march_cull)) != RT_OK) return bail(rc);

    // conservative cull tree (rt_cull.cuh)
    {
        CullTree ct = cull_build(d->inverse, d->kind, (int)n, getenv("RT_B200_NO_CULL") != nullptr,
                                 getenv("RT_B200_NO_CULL_TREE") != nullptr || getenv("RT_B200_NO_CULL") != nullptr, d->params);
        sc->ds.n_roots = ct.n_roots;
        sc->ds.n_upper = ct.n_upper;
        for (int l = 0; l <= RT_CULL_UPPER_MAX; l++) sc->ds.upper_off[l] = ct.upper_off[l];
        if ((rc = upload(sc, ct.upper.data(), ct.upper.size(), &sc->ds.cupper)) != RT_OK) return bail(rc);
        sc->ds.n_groups = ct.n_groups;
        sc->ds.n_flat = ct.n_flat;
        sc->ds.n_flat_real = ct.n_flat_real;
        if ((rc = upload(sc, ct.table.data(), ct.table.size(), &sc->ds.ctab)) != RT_OK) return bail(rc);
        if ((rc = upload(sc, ct.ids.data(), ct.ids.size(), &sc->ds.cids)) != RT_OK) return bail(rc);
        if ((rc = upload(sc, ct.leaf.data(), ct.leaf.size(), &sc->ds.cull)) != RT_OK) return bail(rc);
        if ((rc = upload(sc, ct.group_of.data(), ct.group_of.size(), &sc->ds.cull_group)) != RT_OK) return bail(rc);
        // the flat list's shapes as self-contained records (rt_scene.cuh, FlatRec): inverse rows, Rectangle
        // bounds, index and kind side by side, so that the exact test of flat entry j starts from one address
        // known in advance instead of the chain cids[j] -> kind[id] -> inv[12 id] of dependent loads
        sc->ds.n_frec = 0;
        sc->ds.frec = nullptr;
        if (ct.n_flat_real > 0 && ct.n_flat_real <= RT_FLAT_REC_MAX && !getenv("RT_B200_NO_FLAT_REC")) {
            std::vector<double> frec((size_t)RT_FLAT_REC * ct.n_flat_real, 0.0);
            for (int k = 0; k < ct.n_flat_real; k++) {
                const int id = ct.ids[(size_t)RT_CULL_GROUP * ct.n_groups + k];
                double* r = frec.data() + (size_t)RT_FLAT_REC * k;
                for (int j = 0; j < 12; j++) r[j] = d->inverse[(size_t)12 * id + j];
                for (int j = 0; j < 4; j++) r[12 + j] = d->params[(size_t)RT_SHAPE_PARAMS * id + j];
                const int tag[2] = {id, (int)d->kind[id]};
                memcpy(r + 16, tag, sizeof tag);
            }
            if ((rc = upload(sc, frec.data(), frec.size(), &sc->ds.frec)) != RT_OK) return bail(rc);
            sc->ds.n_frec = ct.n_flat_real;
        }
    }
    // shared-memory staging: 16 B per table entry + the flat list's records
    sc->smem_bytes = (size_t)sc->ds.ctab_entries() * sizeof(float4) + (size_t)sc->ds.n_frec * RT_FLAT_REC * sizeof(double);
    sc->use_smem = n > 0 && sc->smem_bytes > 0 && sc->smem_bytes <= sc->smem_optin;
    if (!sc->use_smem) sc->smem_bytes = 0;
    if (sc->smem_bytes > 48 * 1024) {
        cudaFuncSetAttribute(k_intersect_batch<false, RT_ISECT_BRUTE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_intersect_batch<true, RT_ISECT_BRUTE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_intersect_batch<false, RT_ISECT_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_intersect_batch<true, RT_ISECT_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_intersect_batch<false, RT_ISECT_VERIFY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_bounce<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_bounce<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_extend<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_extend<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_extend<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
        cudaFuncSetAttribute(k_extend<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_bytes);
    }
    // persistent grid: a whole number of CTAs per SM
    int per_sm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_bounce<false>, 256, sc->smem_bytes);
    if (per_sm < 1) per_sm = 1;
    sc->grid = sc->n_sm * per_sm;
    auto occ_grid = [&](auto kernel, int threads, size_t smem) {
        int b = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, threads, smem);
        return sc->n_sm * std::max(b, 1);
    };
    sc->grid_extend = occ_grid(k_extend<false, true>, 256, sc->smem_bytes);
    if (const char* tv = getenv("RT_B200_MARCH_TUNE")) {
        int a = 8, b = 8, c2 = 8, g = 0;
        if (sscanf(tv, "%d,%d,%d,%d", &a, &b, &c2, &g) >= 3) sc->march_tune = make_int3(std::max(a, 1), std::max(b, 1), std::max(c2, 1));
        if (g > 0) sc->march_grid_scale = g;
    }
    {
        int per_sm[3] = {1, 1, 1};
        rt_march_occupancy(per_sm, &sc->smem_march3);
        sc->grid_march = std::max(sc->n_sm * per_sm[0] * sc->march_grid_scale / 100, 1);
        sc->grid_march2 = sc->n_sm * per_sm[1];
        sc->grid_march3 = std::max(sc->n_sm * per_sm[2] * sc->march_grid_scale / 100, 1);
    }
    if (const char* tv0 = getenv("RT_B200_MARCH_TUNE0")) {
        int a = 0, b = 0, c2 = 0;
        if (sscanf(tv0, "%d,%d,%d", &a, &b, &c2) == 3) sc->march_tune0 = make_int3(std::max(a, 1), std::max(b, 1), std::max(c2, 1));
    }
    if (const char* mv = getenv("RT_B200_MARCH")) sc->march_version = std::min(std::max(atoi(mv), 1), 3);
    if (getenv("RT_B200_MARCH_V2")) sc->march_version = 2;
    if (const char* mf = getenv("RT_B200_MARCH_FILTER")) sc->march_filter = atoi(mf) != 0;
    if (!sc->march_filter && !getenv("RT_B200_DEFER_BOUND")) sc->defer_bound = false;   // (measured a net loss without the filter)
    if (const char* db = getenv("RT_B200_DEFER_BOUND")) sc->defer_bound = atoi(db) != 0;
    sc->grid_shade = occ_grid(k_shade<false, true>, 256, 0);
    sc->wavefront = sc->ds.n_march <= 32 && !getenv("RT_B200_FUSED_BOUNCE");

    if (cudaMalloc(&sc->d_counters, sizeof(DevCounters)) != cudaSuccess) return bail(fail(RT_ERR_NOMEM, "cudaMalloc failed"));
    cudaMemset(sc->d_counters, 0, sizeof(DevCounters));
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return bail(fail(RT_ERR_CUDA, std::string("scene upload: ") + cudaGetErrorString(e)));
    *out = sc;
    return RT_OK;
}

int rt_scene_create_multi(const rt_scene_desc* d, int n_devices, const int* device_ids, rt_scene** out) {
    if (!out) return fail(RT_ERR_INVALID, "null out pointer");
    *out = nullptr;
    if (n_devices < 1 || !device_ids) return fail(RT_ERR_INVALID, "no devices");
    if (n_devices > 16) return fail(RT_ERR_INVALID, "at most 16 devices");
    for (int a = 0; a < n_devices; a++)
        for (int b = a + 1; b < n_devices; b++)
            if (device_ids[a] == device_ids[b]) return fail(RT_ERR_INVALID, "a device is listed twice");
    rt_scene* sc = nullptr;
    int rc = rt_scene_create(d, device_ids[0], &sc);
    if (rc != RT_OK) return rc;
    for (int k = 1; k < n_devices; k++) {
        rt_scene* peer = nullptr;
        rc = rt_scene_create(d, device_ids[k], &peer);
        if (rc != RT_OK) {
            rt_scene_destroy(sc);
            return rc;
        }
        sc->peers.push_back(peer);
        sc->d_peer_acc.push_back(nullptr);
        sc->peer_acc_cap.push_back(0);
        // direct NVLink path for the accumulator copies where the topology has one (cudaMemcpyPeerAsync stages
        // through the host otherwise); "already enabled" is fine
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, device_ids[0], device_ids[k]) == cudaSuccess && can) {
            cudaSetDevice(device_ids[0]);
            cudaDeviceEnablePeerAccess(device_ids[k], 0);
        }
        if (cudaDeviceCanAccessPeer(&can, device_ids[k], device_ids[0]) == cudaSuccess && can) {
            cudaSetDevice(device_ids[k]);
            cudaDeviceEnablePeerAccess(device_ids[0], 0);
        }
        cudaGetLastError();
        cudaSetDevice(device_ids[k]);   // the event is recorded on the peer's stream
        cudaEvent_t e = nullptr;
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
            rt_scene_destroy(sc);
            return fail(RT_ERR_CUDA, "cudaEventCreate failed");
        }
        sc->ev_peer.push_back(e);
    }
    cudaSetDevice(device_ids[0]);
    *out = sc;
    return RT_OK;
}

int rt_scene_device_count(rt_scene* sc) { return sc ? (int)sc->peers.size() + 1 : 0; }

// make lane i the one the launch code sees (sc->stream, sc->q, ...)
static void bind_lane(rt_scene* sc, int i) {
    if (i == sc->cur_lane) return;
    PathLane& a = sc->lanes[sc->cur_lane];
    a.stream = sc->stream; a.q[0] = sc->q[0]; a.q[1] = sc->q[1]; a.hq = sc->hq; a.d_radiance = sc->d_radiance;
    a.d_counts = sc->d_counts; a.d_march_state = sc->d_march_state; a.qallocs.swap(sc->qallocs);
    a.path_capacity = sc->path_capacity;
    PathLane& b = sc->lanes[i];
    sc->stream = b.stream; sc->q[0] = b.q[0]; sc->q[1] = b.q[1]; sc->hq = b.hq; sc->d_radiance = b.d_radiance;
    sc->d_counts = b.d_counts; sc->d_march_state = b.d_march_state; sc->qallocs.swap(b.qallocs);
    sc->path_capacity = b.path_capacity;
    sc->cur_lane = i;
}

static void free_lane_buffers(rt_scene* sc) {  // of the bound lane
    for (void* p : sc->qallocs) cudaFree(p);
    sc->qallocs.clear();
    cudaFree(sc->d_radiance); sc->d_radiance = nullptr;
    cudaFree(sc->d_counts); sc->d_counts = nullptr;
    cudaFree(sc->d_march_state); sc->d_march_state = nullptr;
    sc->path_capacity = 0;
}

static void free_render_buffers(rt_scene* sc) {
    for (int l = RT_MAX_LANES - 1; l >= 0; l--) {
        bind_lane(sc, l);
        free_lane_buffers(sc);
    }
    cudaFree(sc->d_accum); sc->d_accum = nullptr;
    cudaFree(sc->d_frame); sc->d_frame = nullptr;
    sc->frame_capacity = 0;
    for (Batch& b : sc->batches) cudaEventDestroy(b.done);
    sc->batches.clear();
}

void rt_scene_destroy(rt_scene* sc) {
    if (!sc) return;
    for (rt_scene* peer : sc->peers) rt_scene_destroy(peer);
    sc->peers.clear();
    cudaSetDevice(sc->device);
    for (Acc* a : sc->d_peer_acc) cudaFree(a);
    for (cudaEvent_t e : sc->ev_peer) cudaEventDestroy(e);
    if (sc->ev_multi_done) cudaEventDestroy(sc->ev_multi_done);
    cudaFree(sc->d_full_frame);
    cudaFree(sc->d_tone_in);
    cudaFree(sc->d_tone_out);
    cudaFree(sc->d_group_off);
    cudaFree(sc->d_group_pix);
    cudaFree(sc->d_group_means);
    cudaFree(sc->d_group_rays);
    cudaFree(sc->d_moments);
    cudaFree(sc->d_plist);
    cudaFree(sc->d_live);
    cudaFree(sc->d_pix_counts);
    if (sc->host_stage) cudaFreeHost(sc->host_stage);
    bind_lane(sc, 0);
    for (int l = 0; l < RT_MAX_LANES; l++)
        if (sc->lanes[l].stream) cudaStreamSynchronize(l == 0 ? sc->stream : sc->lanes[l].stream);
    free_render_buffers(sc);
    bind_lane(sc, 0);
    for (int l = 1; l < RT_MAX_LANES; l++) {
        if (sc->lanes[l].stream) cudaStreamDestroy(sc->lanes[l].stream);
        if (sc->lanes[l].done) cudaEventDestroy(sc->lanes[l].done);
    }
    for (void* p : sc->allocs) cudaFree(p);
    cudaFree(sc->d_counters);
    for (cudaEvent_t e : sc->ev_pool) cudaEventDestroy(e);
    if (sc->ev_a) cudaEventDestroy(sc->ev_a);
    if (sc->ev_b) cudaEventDestroy(sc->ev_b);
    if (sc->ev_frame_start) cudaEventDestroy(sc->ev_frame_start);
    if (sc->ev_frame_stop) cudaEventDestroy(sc->ev_frame_stop);
    if (sc->ev_group_in) cudaEventDestroy(sc->ev_group_in);
    if (sc->ev_group_start) cudaEventDestroy(sc->ev_group_start);
    if (sc->ev_group_done) cudaEventDestroy(sc->ev_group_done);
    if (sc->ev_adaptive_fork) cudaEventDestroy(sc->ev_adaptive_fork);
    if (sc->stream) cudaStreamDestroy(sc->stream);
    if (sc->copy_stream) cudaStreamDestroy(sc->copy_stream);
    delete sc;
}

// ---- batched nearest hit -----------------------------------------------------------------------
int rt_intersect_batch_device(rt_scene* sc, const rt_ray* d_rays, uint64_t n, double t_min, double t_max, int mode,
                              int32_t* d_idx, double* d_t, rt_vec3* d_normal, rt_vec3* d_point, double* d_uv,
                              uint8_t* d_ff, void* stream) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (mode != RT_ISECT_BRUTE && mode != RT_ISECT_FAST && mode != RT_ISECT_VERIFY) return fail(RT_ERR_INVALID, "unknown intersect mode");
    if (n == 0) return RT_OK;
    if (!d_rays) return fail(RT_ERR_INVALID, "null rays");
    CU(cudaSetDevice(sc->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : sc->stream;
    uint64_t want = (n + 255) / 256;
    int grid = (int)std::min<uint64_t>(want, (uint64_t)sc->grid);
#define RT_LAUNCH_ISECT(C_, M_)                                                                                  \
    k_intersect_batch<C_, M_><<<grid, 256, sc->smem_bytes, st>>>(sc->ds, sc->use_smem, d_rays, n, t_min, t_max, d_idx, \
                                                                 d_t, d_normal, d_point, d_uv, d_ff, sc->d_counters)
    if (mode == RT_ISECT_VERIFY) {
        RT_LAUNCH_ISECT(false, RT_ISECT_VERIFY);
    } else if (sc->counters_on) {
        if (mode == RT_ISECT_FAST) RT_LAUNCH_ISECT(true, RT_ISECT_FAST); else RT_LAUNCH_ISECT(true, RT_ISECT_BRUTE);
    } else {
        if (mode == RT_ISECT_FAST) RT_LAUNCH_ISECT(false, RT_ISECT_FAST); else RT_LAUNCH_ISECT(false, RT_ISECT_BRUTE);
    }
#undef RT_LAUNCH_ISECT
    sc->launches++;
    CU(cudaGetLastError());
    return RT_OK;
}

int rt_intersect_batch(rt_scene* sc, const rt_ray* rays, uint64_t n, double t_min, double t_max, int mode,
                       int32_t* idx, double* t, rt_vec3* normal, rt_vec3* point, double* uv, uint8_t* ff) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (n == 0) return RT_OK;
    if (!rays) return fail(RT_ERR_INVALID, "null rays");
    CU(cudaSetDevice(sc->device));
    rt_ray* d_rays = nullptr;
    int32_t* d_idx = nullptr;
    double *d_t = nullptr, *d_uv = nullptr;
    rt_vec3 *d_n = nullptr, *d_p = nullptr;
    uint8_t* d_ff = nullptr;
    int rc = RT_OK;
    auto cleanup = [&]() {
        cudaFree(d_rays); cudaFree(d_idx); cudaFree(d_t); cudaFree(d_uv); cudaFree(d_n); cudaFree(d_p); cudaFree(d_ff);
    };
#define CUX(call)                                                                             \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            cleanup();                                                                        \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));     \
        }                                                                                     \
    } while (0)
    CUX(cudaMalloc(&d_rays, n * sizeof(rt_ray)));
    if (idx) CUX(cudaMalloc(&d_idx, n * sizeof(int32_t)));
    if (t) CUX(cudaMalloc(&d_t, n * sizeof(double)));
    if (uv) CUX(cudaMalloc(&d_uv, 2 * n * sizeof(double)));
    if (normal) CUX(cudaMalloc(&d_n, n * sizeof(rt_vec3)));
    if (point) CUX(cudaMalloc(&d_p, n * sizeof(rt_vec3)));
    if (ff) CUX(cudaMalloc(&d_ff, n));
    CUX(cudaMemcpyAsync(d_rays, rays, n * sizeof(rt_ray), cudaMemcpyHostToDevice, sc->stream));
    CUX(cudaEventRecord(sc->ev_a, sc->stream));
    rc = rt_intersect_batch_device(sc, d_rays, n, t_min, t_max, mode, d_idx, d_t, d_n, d_p, d_uv, d_ff, sc->stream);
    if (rc != RT_OK) {
        cleanup();
        return rc;
    }
    CUX(cudaEventRecord(sc->ev_b, sc->stream));
    if (idx) CUX(cudaMemcpyAsync(idx, d_idx, n * sizeof(int32_t), cudaMemcpyDeviceToHost, sc->stream));
    if (t) CUX(cudaMemcpyAsync(t, d_t, n * sizeof(double), cudaMemcpyDeviceToHost, sc->stream));
    if (uv) CUX(cudaMemcpyAsync(uv, d_uv, 2 * n * sizeof(double), cudaMemcpyDeviceToHost, sc->stream));
    if (normal) CUX(cudaMemcpyAsync(normal, d_n, n * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->stream));
    if (point) CUX(cudaMemcpyAsync(point, d_p, n * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->stream));
    if (ff) CUX(cudaMemcpyAsync(ff, d_ff, n, cudaMemcpyDeviceToHost, sc->stream));
    CUX(cudaStreamSynchronize(sc->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, sc->ev_a, sc->ev_b);
    sc->last_intersect_ms = ms;
    cleanup();
#undef CUX
    return RT_OK;
}

// ---- rendering ---------------------------------------------------------------------------------
static RayCasterDev make_raycaster(const rt_camera& cam, rt_image_params img) {
    // MultisamplerRayCaster::new, src/camera/ray_caster.rs:30-48 (host FP64: needs libm tan).
    // This file is compiled with -fmad=false, which also governs host code generated by nvcc's
    // host compiler pass?  No: host code goes to g++, so -ffp-contract=off is passed via -Xcompiler.
    auto V = [](rt_vec3 a) { return D3{a.x, a.y, a.z}; };
    D3 pos = V(cam.position), dir = V(cam.direction), right = V(cam.right), up = V(cam.up);
    D3 center = {pos.x + dir.x * cam.focal_length, pos.y + dir.y * cam.focal_length, pos.z + dir.z * cam.focal_length};
    double aspect_ratio = (double)img.width / (double)img.height;
    double viewport_width = tan(cam.fov_rad / 2.0) * cam.focal_length * 2.0;
    double viewport_height = viewport_width / aspect_ratio;
    double hw = viewport_width / 2.0, hh = viewport_height / 2.0;
    RayCasterDev rc;
    rc.left_top = D3{(center.x - hw * right.x) + hh * up.x, (center.y - hw * right.y) + hh * up.y,
                     (center.z - hw * right.z) + hh * up.z};
    rc.pixel_resolution = viewport_width / (double)img.width;
    rc.camera_position = pos;
    rc.camera_right = right;
    rc.camera_up = up;
    return rc;
}

static cudaEvent_t pool_event(rt_scene* sc) {
    if (sc->ev_used == sc->ev_pool.size()) {
        cudaEvent_t e = nullptr;
        cudaEventCreate(&e);
        sc->ev_pool.push_back(e);
    }
    return sc->ev_pool[sc->ev_used++];
}
struct KernelSpan {  // RAII: records an event pair around one launch when kernel timing is on
    rt_scene* sc;
    int cls;
    cudaEvent_t a = nullptr;
    KernelSpan(rt_scene* s, int c) : sc(s), cls(c) {
        sc->launches++;
        if (!sc->ktiming) return;
        a = pool_event(sc);
        cudaEventRecord(a, sc->stream);
    }
    ~KernelSpan() {
        if (!a) return;
        cudaEvent_t b = pool_event(sc);
        cudaEventRecord(b, sc->stream);
        sc->spans.push_back({cls, a, b});
    }
};
static void resolve_spans(rt_scene* sc) {  // the stream must have passed every recorded event
    for (auto& sp : sc->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
            sc->ms_cls[sp.cls] += ms;
            sc->n_cls[sp.cls]++;
        }
    }
    cudaGetLastError();
    sc->spans.clear();
    sc->ev_used = 0;
}

static int alloc_queue(rt_scene* sc, PathQueue& q, uint64_t cap) {
    double** d[9] = {&q.ox, &q.oy, &q.oz, &q.dx, &q.dy, &q.dz, &q.bx, &q.by, &q.bz};
    for (int k = 0; k < 9; k++) {
        void* p = nullptr;
        CU(cudaMalloc(&p, cap * sizeof(double)));
        sc->qallocs.push_back(p);
        *d[k] = (double*)p;
    }
    void* p = nullptr;
    CU(cudaMalloc(&p, cap * sizeof(uint32_t)));
    sc->qallocs.push_back(p);
    q.pid = (uint32_t*)p;
    return RT_OK;
}


// enqueue the bounce loop for paths already in q[0] (count in d_counts[0]); no host sync
static void launch_bounces(rt_scene* sc, uint32_t max_depth, uint64_t seed, const RaygenArgs* raygen = nullptr) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    for (uint32_t level = 0; level <= max_depth; level++) {
        PathQueue& in = sc->q[level & 1];
        PathQueue& out = sc->q[(level + 1) & 1];
        uint32_t* cnt_in = sc->d_counts + level;
        uint32_t* cnt_out = sc->d_counts + level + 1;
        uint32_t* mcount = sc->d_counts + RT_CNT_MARCH + level;
        uint32_t* rcount = sc->d_counts + RT_CNT_REPLAY + level;
        if (!sc->wavefront) {
            KernelSpan span(sc, RT_KCLASS_EXTEND);
            if (sc->counters_on)
                k_bounce<true><<<sc->grid, 256, sc->smem_bytes, sc->stream>>>(sc->ds, sc->use_smem, in, cnt_in, out, cnt_out, level,
                                                                              max_depth, sc->hq.key, k0, k1, sc->d_radiance,
                                                                              sc->d_counters);
            else
                k_bounce<false><<<sc->grid, 256, sc->smem_bytes, sc->stream>>>(sc->ds, sc->use_smem, in, cnt_in, out, cnt_out, level,
                                                                               max_depth, sc->hq.key, k0, k1, sc->d_radiance,
                                                                               sc->d_counters);
            continue;
        }
        {
            KernelSpan span(sc, RT_KCLASS_EXTEND);
            const bool gen = level == 0 && raygen != nullptr;   // the frame's primary rays are generated in place
            RaygenArgs rg{};
            if (gen) rg = *raygen;
#define RT_LAUNCH_EXTEND(C_, G_)                                                                                        \
    k_extend<C_, G_><<<sc->grid_extend, 256, sc->smem_bytes, sc->stream>>>(sc->ds, sc->use_smem, in, cnt_in, sc->hq, mcount, \
                                                                           rcount, sc->d_counters, level == max_depth,     \
                                                                           sc->defer_bound, rg)
            if (sc->counters_on) {
                if (gen) RT_LAUNCH_EXTEND(true, true); else RT_LAUNCH_EXTEND(true, false);
            } else {
                if (gen) RT_LAUNCH_EXTEND(false, true); else RT_LAUNCH_EXTEND(false, false);
            }
#undef RT_LAUNCH_EXTEND
        }
        if (sc->ds.n_march > 0) {
            KernelSpan span(sc, RT_KCLASS_MARCH);
            if (sc->march_filter) {   // the miss proof for every queued (ray, shape) pair, with full warps
                MarchLaunch fl;
                fl.ds = sc->ds; fl.in = in; fl.hq = sc->hq; fl.march_count = mcount; fl.counters = sc->d_counters;
                fl.count = sc->counters_on; fl.stream = sc->stream; fl.grid_filter = sc->n_sm * 8;
                fl.filtered_count = sc->d_counts + RT_CNT_FILTERED + level;
                rt_launch_march_filter(fl);
                sc->launches++;
            }
            // the marching kernels read the compacted queue the filter wrote
            HitQueue mhq = sc->hq;
            const uint32_t* mq_count = mcount;
            if (sc->march_filter) {
                mhq.mq_slot = sc->hq.fq_slot;
                mhq.mq_mask = sc->hq.fq_mask;
                mq_count = sc->d_counts + RT_CNT_FILTERED + level;
            }
            for (int kind = 0; kind < 6; kind++) {
                if (!sc->kind_mask[kind]) continue;
                uint32_t* head = sc->d_counts + RT_CNT_HEAD + kind * RT_MAX_LEVELS + level;
                MarchLaunch ml;
                ml.ds = sc->ds; ml.kind = kind; ml.kind_mask = sc->kind_mask[kind]; ml.in = in; ml.hq = mhq;
                ml.march_count = mq_count; ml.head = head; ml.counters = sc->d_counters; ml.count = sc->counters_on;
                ml.stream = sc->stream; ml.version = sc->march_version; ml.grid1 = sc->grid_march; ml.grid2 = sc->grid_march2;
                ml.grid3 = sc->grid_march3; ml.smem3 = sc->smem_march3; ml.tune = level == 0 ? sc->march_tune0 : sc->march_tune; ml.march_state = sc->d_march_state;
                ml.prefiltered = sc->march_filter; ml.grid_filter = 0;
                rt_launch_march(ml);
                sc->launches++;
            }
            sc->launches--;  // the span already counted one launch
        }
        {   // degenerate rays (rare; the kernel exits at once when its queue is empty)
            KernelSpan span(sc, RT_KCLASS_MARCH);
            k_replay<<<sc->n_sm, 128, 0, sc->stream>>>(sc->ds, in, sc->hq, rcount);
        }
        {
            KernelSpan span(sc, RT_KCLASS_SHADE);
            // the binned variant only where it has something to sort: several shade keys in the scene, and not at the
            // last level (any hit is black there)
            const bool binned = sc->shade_binned && level < max_depth;
#define RT_LAUNCH_SHADE(C_, B_)                                                                                              \
    k_shade<C_, B_><<<sc->grid_shade, 256, 0, sc->stream>>>(sc->ds, in, cnt_in, sc->hq, out, cnt_out, level, max_depth, sc->map, \
                                                            0ull, 1u, k0, k1, sc->d_radiance)
            if (sc->counters_on) {
                if (binned) RT_LAUNCH_SHADE(true, true); else RT_LAUNCH_SHADE(true, false);
            } else {
                if (binned) RT_LAUNCH_SHADE(false, true); else RT_LAUNCH_SHADE(false, false);
            }
#undef RT_LAUNCH_SHADE
        }
    }
}

static int ensure_path_buffers(rt_scene* sc, uint64_t need_paths) {
    if (sc->path_capacity >= need_paths) return RT_OK;  // (of the bound lane)
    for (void* p : sc->qallocs) cudaFree(p);
    sc->qallocs.clear();
    cudaFree(sc->d_radiance); sc->d_radiance = nullptr;
    sc->path_capacity = 0;
    int rc;
    if ((rc = alloc_queue(sc, sc->q[0], need_paths)) != RT_OK) return rc;
    if ((rc = alloc_queue(sc, sc->q[1], need_paths)) != RT_OK) return rc;
    CU(cudaMalloc(&sc->d_radiance, need_paths * sizeof(float4)));
    {
        void* p = nullptr;
        CU(cudaMalloc(&p, need_paths * sizeof(double))); sc->qallocs.push_back(p); sc->hq.t = (double*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(int32_t))); sc->qallocs.push_back(p); sc->hq.index = (int32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint32_t))); sc->qallocs.push_back(p); sc->hq.mq_slot = (uint32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint32_t))); sc->qallocs.push_back(p); sc->hq.mq_mask = (uint32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint32_t))); sc->qallocs.push_back(p); sc->hq.fq_slot = (uint32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint32_t))); sc->qallocs.push_back(p); sc->hq.fq_mask = (uint32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint32_t))); sc->qallocs.push_back(p); sc->hq.rq_slot = (uint32_t*)p;
        CU(cudaMalloc(&p, need_paths * sizeof(uint2))); sc->qallocs.push_back(p); sc->hq.key = (uint2*)p;
    }
    if (!sc->d_counts) CU(cudaMalloc(&sc->d_counts, RT_CNT_WORDS * sizeof(uint32_t)));
    if (!sc->d_march_state && sc->ds.n_march > 0 && sc->march_version == 2)
        CU(cudaMalloc(&sc->d_march_state, rt_march2_state_bytes(sc->grid_march2)));
    sc->path_capacity = need_paths;
    return RT_OK;
}

static int render_start_single(rt_scene* sc, const rt_camera* cam, const rt_render_params* p,
                               const rt_adaptive_params* ap = nullptr);
static int render_start_multi(rt_scene* sc, const rt_camera* cam, const rt_render_params* p);

int rt_render_start(rt_scene* sc, const rt_camera* cam, const rt_render_params* p) {
    if (!sc || !cam || !p) return fail(RT_ERR_INVALID, "null argument");
    // a handle over several devices shards a WHOLE-frame request over them; an explicitly sharded request
    // (one process per GPU on top of it) renders its shard on the first device as always
    if (!sc->peers.empty() && p->shard_count <= 1) return render_start_multi(sc, cam, p);
    sc->multi_active = false;
    return render_start_single(sc, cam, p);
}

// One refinement pass of an adaptive frame: the listed pixels hold n samples and get m more, B pixels per batch,
// planned for the worst case of every owned pixel listed (nb batches; the ones past the list's end exit at once).
struct RefinePass {
    uint32_t n, m;
    uint64_t B, nb;
};

// ap != NULL: an adaptive frame (rt_render_start_adaptive, validated there).  Pass 0 is the frame path with
// min_samples samples (k_resolve<true> also writes the moments); the refinement passes follow in the same enqueue.
static int render_start_single(rt_scene* sc, const rt_camera* cam, const rt_render_params* p, const rt_adaptive_params* ap) {
    if (!sc || !cam || !p) return fail(RT_ERR_INVALID, "null argument");
    if (p->image.width == 0 || p->image.height == 0 || p->samples_number == 0)
        return fail(RT_ERR_INVALID, "empty image or zero samples");
    if (p->max_depth > RT_MAX_LEVELS - 2) return fail(RT_ERR_INVALID, "max_depth too large (limit 62)");
    uint32_t shard_count = p->shard_count ? p->shard_count : 1;
    if (p->shard_index >= shard_count) return fail(RT_ERR_INVALID, "shard_index >= shard_count");
    if (shard_count > 16) return fail(RT_ERR_INVALID, "at most 16 shards");
    if ((uint64_t)p->image.width * p->image.height > 0xFFFFFFFFull) return fail(RT_ERR_INVALID, "image too large");
    {
        rt_render_params pp = *p;
        pp.shard_count = shard_count;
        if (!tile_fits(make_shard_map(pp, p->shard_index))) return fail(RT_ERR_INVALID, "tile_width * tile_height >= 2^32");
    }
    CU(cudaSetDevice(sc->device));
    if (sc->rendering) rt_render_stop(sc);

    // progressive accumulation: this frame adds its samples to the previous ones when it is the same frame
    // (image, sharding, depth, seed, camera) and nothing was abandoned; otherwise it starts afresh
    uint32_t sample_base = 0;
    if (!ap && sc->accumulate && sc->accumulated_spp > 0 && sc->wavefront && memcmp(&sc->accum_cam, cam, sizeof *cam) == 0 &&
        sc->accum_rp.image.width == p->image.width && sc->accum_rp.image.height == p->image.height &&
        sc->accum_rp.max_depth == p->max_depth && sc->accum_rp.seed == p->seed &&
        (sc->accum_rp.shard_count ? sc->accum_rp.shard_count : 1) == shard_count &&
        sc->accum_rp.shard_index == p->shard_index && sc->accum_rp.tile_width == p->tile_width &&
        sc->accum_rp.tile_height == p->tile_height &&
        (uint64_t)sc->accumulated_spp + p->samples_number <= 0xFFFFFFFFull)
        sample_base = sc->accumulated_spp;
    sc->accumulated_spp = 0;  // until this frame is enqueued (an abandoned frame breaks the chain)
    sc->adaptive_frame = false;
    sc->rp = *p;
    sc->rp.shard_count = shard_count;
    sc->map = make_shard_map(sc->rp, p->shard_index);
    sc->owned_pixels = owned_tiles(sc->map) * sc->map.tile_pixels();

    const uint32_t spp = ap ? ap->min_samples : p->samples_number;
    uint64_t cap_paths = env_size("RT_B200_BATCH_PATHS", (size_t)1 << 23);
    // adaptive: the refinement passes n_k -> n_k + min(n_k, samples_number - n_k), B_k = max(1, cap / m_k) pixels per batch
    std::vector<RefinePass> refine;
    uint64_t refine_batches = 0, refine_paths = 0;
    if (ap) {
        const uint64_t cap = std::min<uint64_t>(std::max<uint64_t>(cap_paths, 1), 0xFFFFFFF0ull);
        for (uint32_t n = ap->min_samples; n < p->samples_number;) {
            const uint32_t m = std::min(n, p->samples_number - n);
            const uint64_t B = std::min<uint64_t>(std::max<uint64_t>(1, cap / m), std::max<uint64_t>(sc->owned_pixels, 1));
            const uint64_t nb = (sc->owned_pixels + B - 1) / B;
            refine.push_back({n, m, B, nb});
            refine_batches = std::max(refine_batches, nb);
            refine_paths = std::max(refine_paths, B * m);
            n += m;
        }
    }
    uint64_t px_per_batch = std::max<uint64_t>(1, cap_paths / spp);
    // batches alternate between lanes (streams); per-kernel timing wants the launches back to back
    int lanes_used = sc->ktiming ? 1 : sc->n_lanes;
    if (!sc->lanes_from_env && lanes_used > 2) {
        const uint64_t full = (std::max<uint64_t>(sc->owned_pixels, 1) + px_per_batch - 1) / px_per_batch;
        if (full < 6) lanes_used = 2;
    }
    if (lanes_used > 1) {  // a frame of one batch is split when each part still fills the GPU
        uint64_t split = (std::max<uint64_t>(sc->owned_pixels, 1) + lanes_used - 1) / lanes_used;
        if (split * spp >= ((uint64_t)1 << 20)) px_per_batch = std::min(px_per_batch, split);
    }
    px_per_batch = std::min<uint64_t>(px_per_batch, std::max<uint64_t>(sc->owned_pixels, 1));
    if (px_per_batch * spp > 0xFFFFFFF0ull) return fail(RT_ERR_INVALID, "samples_number too large for one batch");
    const uint64_t n_batches = (sc->owned_pixels + px_per_batch - 1) / px_per_batch;
    lanes_used = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)lanes_used, std::max(n_batches, refine_batches)));
    int rc = RT_OK;
    for (int l = 0; l < lanes_used && rc == RT_OK; l++) {
        bind_lane(sc, l);
        rc = ensure_path_buffers(sc, std::max<uint64_t>(px_per_batch * spp, refine_paths));
    }
    bind_lane(sc, 0);
    if (rc != RT_OK) return rc;
    if (sc->frame_capacity < sc->owned_pixels) {
        cudaFree(sc->d_accum); cudaFree(sc->d_frame);
        sc->d_accum = nullptr; sc->d_frame = nullptr; sc->frame_capacity = 0;
        CU(cudaMalloc(&sc->d_accum, std::max<uint64_t>(sc->owned_pixels, 1) * sizeof(Acc)));
        CU(cudaMalloc(&sc->d_frame, std::max<uint64_t>(sc->owned_pixels, 1) * sizeof(rt_vec3)));
        sc->frame_capacity = sc->owned_pixels;
    }
    if (ap) {
        if ((rc = ensure_device_array(sc->d_moments, sc->moments_cap, sc->owned_pixels)) != RT_OK) return rc;
        if ((rc = ensure_device_array(sc->d_plist, sc->plist_cap, sc->owned_pixels)) != RT_OK) return rc;
        if ((rc = ensure_device_array(sc->d_live, sc->live_cap, std::max<uint64_t>(refine.size(), 1))) != RT_OK) return rc;
    }
    for (Batch& b : sc->batches) cudaEventDestroy(b.done);
    sc->batches.clear();
    sc->delivered = 0;
    sc->spans.clear();
    sc->ev_used = 0;

    RayCasterDev rcd = make_raycaster(*cam, p->image);
    uint32_t k0 = (uint32_t)p->seed, k1 = (uint32_t)(p->seed >> 32);
    auto enqueue = [&]() -> int {
        CU(cudaEventRecord(sc->ev_frame_start, sc->stream));  // lane 0 = the main stream
        for (int l = 1; l < lanes_used; l++) CU(cudaStreamWaitEvent(sc->lanes[l].stream, sc->ev_frame_start, 0));
        if (ap) CU(cudaMemsetAsync(sc->d_live, 0, std::max<size_t>(refine.size(), 1) * sizeof(uint32_t), sc->stream));
        uint64_t batch_no = 0;
        for (uint64_t first = 0; first < sc->owned_pixels; first += px_per_batch, batch_no++) {
            bind_lane(sc, (int)(batch_no % (uint64_t)lanes_used));
            uint32_t npx = (uint32_t)std::min<uint64_t>(px_per_batch, sc->owned_pixels - first);
            CU(cudaMemsetAsync(sc->d_counts, 0, RT_CNT_WORDS * sizeof(uint32_t), sc->stream));
            if (sc->wavefront) {   // primary rays are generated inside the level-0 k_extend
                RaygenArgs rg;
                rg.rc = rcd; rg.map = sc->map; rg.first_owned = first; rg.n_paths = npx * spp; rg.spp = spp;
                rg.k0 = k0; rg.k1 = k1; rg.sample_base = sample_base; rg.radiance = sc->d_radiance; rg.count_out = sc->d_counts;
                launch_bounces(sc, p->max_depth, p->seed, &rg);
            } else {
                {
                    KernelSpan span(sc, RT_KCLASS_RAYGEN);
                    k_raygen<<<sc->grid, 256, 0, sc->stream>>>(rcd, sc->map, first, npx, spp, k0, k1, sc->q[0], sc->d_counts, sc->d_radiance, sc->hq.key, sample_base);
                }
                launch_bounces(sc, p->max_depth, p->seed);
            }
            {
                KernelSpan span(sc, RT_KCLASS_RESOLVE);
                if (ap)
                    k_resolve<true><<<(npx + 255) / 256, 256, 0, sc->stream>>>(sc->d_radiance, npx, spp, first, sc->d_accum,
                                                                             sc->d_frame, false, sc->d_moments);
                else
                    k_resolve<false><<<(npx + 255) / 256, 256, 0, sc->stream>>>(sc->d_radiance, npx, spp, first, sc->d_accum,
                                                                              sc->d_frame, sample_base != 0, nullptr);
            }
            if (ap) continue;   // an adaptive frame is delivered whole, after its last pass
            Batch b;
            b.first_owned = first;
            b.n_pixels = npx;
            CU(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
            CU(cudaEventRecord(b.done, sc->stream));
            sc->batches.push_back(b);
            sc->paths += (uint64_t)npx * spp;
        }
        // adaptive refinement passes: all lanes join the main stream, k_adaptive_select lists the pixels that go on,
        // the lanes fork again and run the pass's batches.  Nothing waits on the host.
        const uint32_t width = sc->map.width;
        for (size_t k = 0; k < refine.size(); k++) {
            const RefinePass& P = refine[k];
            bind_lane(sc, 0);
            for (int l = 1; l < lanes_used; l++) {
                CU(cudaEventRecord(sc->lanes[l].done, sc->lanes[l].stream));
                CU(cudaStreamWaitEvent(sc->stream, sc->lanes[l].done, 0));
            }
            {
                KernelSpan span(sc, RT_KCLASS_RESOLVE);
                const unsigned grid = (unsigned)std::min<uint64_t>((sc->owned_pixels + 255) / 256, (uint64_t)sc->n_sm * 8);
                k_adaptive_select<<<std::max(grid, 1u), 256, 0, sc->stream>>>(sc->d_accum, sc->d_moments, (uint32_t)sc->owned_pixels,
                                                                              (double)P.n, ap->rel_error, ap->abs_error,
                                                                              sc->d_plist, sc->d_live + k);
            }
            CU(cudaEventRecord(sc->ev_adaptive_fork, sc->stream));
            for (int l = 1; l < lanes_used; l++) CU(cudaStreamWaitEvent(sc->lanes[l].stream, sc->ev_adaptive_fork, 0));
            const uint32_t B = (uint32_t)P.B;
            const unsigned grid_gen = (unsigned)std::min<uint64_t>((P.B * P.m + 255) / 256, (uint64_t)sc->n_sm * 16);
            for (uint64_t j = 0; j < P.nb; j++) {
                bind_lane(sc, (int)(j % (uint64_t)lanes_used));
                CU(cudaMemsetAsync(sc->d_counts, 0, RT_CNT_WORDS * sizeof(uint32_t), sc->stream));
                {
                    KernelSpan span(sc, RT_KCLASS_RAYGEN);
                    k_raygen_list<<<grid_gen, 256, 0, sc->stream>>>(rcd, width, sc->d_plist, sc->d_live + k, (uint32_t)(j * P.B), B,
                                                                    P.m, P.n, k0, k1, sc->q[0], sc->hq.key, sc->d_counts);
                }
                launch_bounces(sc, p->max_depth, p->seed);
                {
                    KernelSpan span(sc, RT_KCLASS_RESOLVE);
                    k_resolve_list<<<(unsigned)((P.B + 255) / 256), 256, 0, sc->stream>>>(
                        sc->d_radiance, sc->d_plist, sc->d_live + k, (uint32_t)(j * P.B), B, P.m, sc->d_accum, sc->d_moments,
                        sc->d_frame);
                }
            }
        }
        bind_lane(sc, 0);
        for (int l = 1; l < lanes_used; l++) {  // the main stream ends the frame after every lane
            CU(cudaEventRecord(sc->lanes[l].done, sc->lanes[l].stream));
            CU(cudaStreamWaitEvent(sc->stream, sc->lanes[l].done, 0));
        }
        if (ap) {   // one delivery unit: the whole frame, once the last pass has resolved
            Batch b;
            b.first_owned = 0;
            b.n_pixels = (uint32_t)sc->owned_pixels;
            CU(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
            CU(cudaEventRecord(b.done, sc->stream));
            sc->batches.push_back(b);
        }
        CU(cudaEventRecord(sc->ev_frame_stop, sc->stream));
        CU(cudaGetLastError());
        return RT_OK;
    };
    rc = enqueue();
    bind_lane(sc, 0);
    if (rc != RT_OK) return rc;
    sc->rendering = true;
    sc->frame_complete = false;
    if (ap) {   // rt_stats.paths grows when the frame completes (the listed counts are known on the device only)
        sc->adaptive_frame = true;
        sc->adaptive_m.assign(1, spp);
        for (const RefinePass& P : refine) sc->adaptive_m.push_back(P.m);
        return RT_OK;
    }
    if (sc->accumulate && sc->wavefront) {  // (enqueued work always runs to completion: rt_render_stop drains it)
        sc->accumulated_spp = sample_base + spp;
        sc->accum_rp = *p;
        sc->accum_cam = *cam;
    }
    return RT_OK;
}

// Whole frame on every device of the handle: device k renders shard k of n (interleaved 32x32 tiles, rotated rows:
// ShardMap), all of them concurrently -- every call below only enqueues -- then each peer's accumulator travels to
// the first device with ONE peer copy on the peer's own stream (so it is ordered behind that shard's last
// k_resolve and the peer is free for its next frame as soon as the copy has left), and k_assemble builds the frame
// behind the events of all copies.  Nothing here waits on the host.
static int render_start_multi(rt_scene* sc, const rt_camera* cam, const rt_render_params* p) {
    if (p->image.width == 0 || p->image.height == 0 || p->samples_number == 0)
        return fail(RT_ERR_INVALID, "empty image or zero samples");
    const uint32_t n_dev = (uint32_t)sc->peers.size() + 1;
    rt_render_params sp = *p;
    sp.shard_count = n_dev;
    if (!sp.tile_width) sp.tile_width = 32;
    if (!sp.tile_height) sp.tile_height = 32;
    const uint64_t n_px = (uint64_t)p->image.width * p->image.height;
    CU(cudaSetDevice(sc->device));
    if (sc->multi_active && sc->ev_multi_done) CU(cudaEventSynchronize(sc->ev_multi_done));   // d_full_frame / staging still in use
    if (sc->full_frame_cap < n_px) {
        cudaFree(sc->d_full_frame);
        sc->d_full_frame = nullptr;
        sc->full_frame_cap = 0;
        CU(cudaMalloc(&sc->d_full_frame, n_px * sizeof(rt_vec3)));
        sc->full_frame_cap = n_px;
    }
    if (!sc->ev_multi_done) CU(cudaEventCreate(&sc->ev_multi_done));
    for (uint32_t k = 1; k < n_dev; k++) {
        const uint64_t need = rt_shard_float4_count(&sp, k);
        if (sc->peer_acc_cap[k - 1] < need) {
            cudaFree(sc->d_peer_acc[k - 1]);
            sc->d_peer_acc[k - 1] = nullptr;
            sc->peer_acc_cap[k - 1] = 0;
            CU(cudaMalloc(&sc->d_peer_acc[k - 1], std::max<uint64_t>(need, 1) * sizeof(Acc)));
            sc->peer_acc_cap[k - 1] = need;
        }
    }
    // enqueue every shard (the peers first: the first device also assembles)
    for (uint32_t k = 1; k < n_dev; k++) {
        rt_scene* peer = sc->peers[k - 1];
        sp.shard_index = k;
        int rc = render_start_single(peer, cam, &sp);
        if (rc != RT_OK) return rc;
        const uint64_t cnt = rt_shard_float4_count(&sp, k);
        if (cnt) CU(cudaMemcpyPeerAsync(sc->d_peer_acc[k - 1], sc->device, peer->d_accum, peer->device, cnt * sizeof(Acc), peer->stream));
        CU(cudaEventRecord(sc->ev_peer[k - 1], peer->stream));
    }
    sp.shard_index = 0;
    int rc = render_start_single(sc, cam, &sp);
    if (rc != RT_OK) return rc;
    CU(cudaSetDevice(sc->device));
    for (uint32_t k = 1; k < n_dev; k++) CU(cudaStreamWaitEvent(sc->stream, sc->ev_peer[k - 1], 0));
    ShardPtrs ptrs;
    for (uint32_t k = 0; k < 16; k++) ptrs.p[k] = k == 0 ? sc->d_accum : k < n_dev ? sc->d_peer_acc[k - 1] : nullptr;
    ShardMap m0 = make_shard_map(sp, 0);
    k_assemble<<<(unsigned)((n_px + 255) / 256), 256, 0, sc->stream>>>(ptrs, m0, sc->d_full_frame);
    sc->launches++;
    CU(cudaEventRecord(sc->ev_multi_done, sc->stream));
    CU(cudaGetLastError());
    sc->multi_active = true;
    sc->multi_rp = *p;
    return RT_OK;
}

int rt_render_set_accumulate(rt_scene* sc, int enabled) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (enabled && !sc->wavefront)
        return fail(RT_ERR_STATE, "progressive accumulation needs the wavefront renderer (at most 32 ray-marched shapes)");
    for (rt_scene* peer : sc->peers) {
        int rc = rt_render_set_accumulate(peer, enabled);
        if (rc != RT_OK) return rc;
    }
    sc->accumulate = enabled != 0;
    sc->accumulated_spp = 0;
    return RT_OK;
}

int rt_render_accumulated_samples(rt_scene* sc, uint32_t* samples) {
    if (!sc || !samples) return fail(RT_ERR_INVALID, "null argument");
    *samples = sc->accumulated_spp;
    return RT_OK;
}

int rt_render_start_adaptive(rt_scene* sc, const rt_camera* cam, const rt_render_params* p, const rt_adaptive_params* ap) {
    if (!sc || !cam || !p || !ap) return fail(RT_ERR_INVALID, "null argument");
    if (!sc->peers.empty()) return fail(RT_ERR_INVALID, "adaptive sampling: not available on a multi-device handle");
    if (p->shard_count > 1) return fail(RT_ERR_INVALID, "adaptive sampling renders whole frames (shard_count 0 or 1)");
    if (ap->min_samples < 2 || ap->min_samples > p->samples_number)
        return fail(RT_ERR_INVALID, "adaptive sampling needs 2 <= min_samples <= samples_number");
    if (!(std::isfinite(ap->rel_error) && ap->rel_error >= 0.0) || !(std::isfinite(ap->abs_error) && ap->abs_error >= 0.0))
        return fail(RT_ERR_INVALID, "adaptive sampling: rel_error and abs_error must be finite and >= 0");
    if (!sc->wavefront)
        return fail(RT_ERR_STATE, "adaptive sampling needs the wavefront renderer (at most 32 ray-marched shapes)");
    sc->multi_active = false;
    return render_start_single(sc, cam, p, ap);
}

int rt_render_pixel_stats(rt_scene* sc, uint32_t* counts, double* moments) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (sc->multi_active) return fail(RT_ERR_STATE, "per-pixel statistics of a multi-device frame are not kept");
    if (sc->rendering) {
        CU(cudaSetDevice(sc->device));
        CU(cudaStreamSynchronize(sc->stream));
        int done = 0;
        int rc = rt_render_poll(sc, nullptr, &done);
        if (rc != RT_OK) return rc;
    }
    if (!sc->frame_complete) return fail(RT_ERR_STATE, "no completed frame");
    if (sc->map.shard_count != 1) return fail(RT_ERR_STATE, "the last frame was one shard of a frame");
    if (moments && !sc->adaptive_frame) return fail(RT_ERR_STATE, "moments are kept for adaptive frames only");
    CU(cudaSetDevice(sc->device));
    const uint64_t n = sc->owned_pixels;   // == width * height: owned order is x + y*width for an unsharded frame
    if (counts && n) {
        int rc = ensure_device_array(sc->d_pix_counts, sc->pix_counts_cap, n);
        if (rc != RT_OK) return rc;
        k_pixel_counts<<<(unsigned)((n + 255) / 256), 256, 0, sc->copy_stream>>>(sc->d_accum, (uint32_t)n, sc->d_pix_counts);
        sc->launches++;
        CU(cudaMemcpyAsync(counts, sc->d_pix_counts, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, sc->copy_stream));
    }
    if (moments && n) CU(cudaMemcpyAsync(moments, sc->d_moments, n * sizeof(double2), cudaMemcpyDeviceToHost, sc->copy_stream));
    const cudaError_t e = cudaStreamSynchronize(sc->copy_stream);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("pixel stats: ") + cudaGetErrorString(e));
    return RT_OK;
}

// copy the owned-order range [q0, q1) of the f64 frame to the caller's x + y*w buffer
static int deliver(rt_scene* sc, uint64_t q0, uint64_t q1, rt_vec3* buffer) {
    if (q1 <= q0) return RT_OK;
    if (sc->map.shard_count == 1) {  // owned order is row-major: one contiguous copy
        CU(cudaMemcpyAsync(buffer + q0, sc->d_frame + q0, (q1 - q0) * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->copy_stream));
        CU(cudaStreamSynchronize(sc->copy_stream));
        return RT_OK;
    }
    // a shard's pixels: pinned staging, then one memcpy per tile row (tile_w contiguous pixels of the caller's frame)
    if (sc->host_stage_cap < q1 - q0) {
        if (sc->host_stage) cudaFreeHost(sc->host_stage);
        sc->host_stage = nullptr;
        sc->host_stage_cap = 0;
        CU(cudaMallocHost(&sc->host_stage, (q1 - q0) * sizeof(rt_vec3)));
        sc->host_stage_cap = q1 - q0;
    }
    CU(cudaMemcpyAsync(sc->host_stage, sc->d_frame + q0, (q1 - q0) * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->copy_stream));
    CU(cudaStreamSynchronize(sc->copy_stream));
    const uint32_t tw = sc->map.tile_w;
    for (uint64_t q = q0; q < q1;) {
        uint32_t x, y;
        const uint64_t run = std::min<uint64_t>(tw - (q % tw), q1 - q);   // to the end of this tile row
        if (sc->map.pixel_of(q, x, y)) {
            const uint64_t keep = std::min<uint64_t>(run, sc->map.width - x);   // clipped border tile
            memcpy(buffer + (size_t)y * sc->map.width + x, sc->host_stage + (q - q0), keep * sizeof(rt_vec3));
        }
        q += run;
    }
    return RT_OK;
}

static int finish_frame(rt_scene* sc);   // bookkeeping of a completed single-device frame

// the frame of a multi-device handle: complete when k_assemble has run; delivered with one contiguous copy
static int render_poll_multi(rt_scene* sc, rt_vec3* buffer, int* done) {
    CU(cudaSetDevice(sc->device));
    cudaError_t e = cudaEventQuery(sc->ev_multi_done);
    if (e == cudaErrorNotReady) {
        *done = 0;
        return RT_OK;
    }
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("render: ") + cudaGetErrorString(e));
    for (rt_scene* peer : sc->peers) {   // their streams are past the peer copy: close their frames
        int rc = finish_frame(peer);
        if (rc != RT_OK) return rc;
    }
    int rc = finish_frame(sc);
    if (rc != RT_OK) return rc;
    CU(cudaSetDevice(sc->device));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, sc->ev_frame_start, sc->ev_multi_done);
    sc->last_frame_ms = ms;
    if (buffer) {
        const uint64_t n_px = (uint64_t)sc->multi_rp.image.width * sc->multi_rp.image.height;
        CU(cudaMemcpyAsync(buffer, sc->d_full_frame, n_px * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->copy_stream));
        CU(cudaStreamSynchronize(sc->copy_stream));
    }
    *done = 1;
    return RT_OK;
}

static int finish_frame(rt_scene* sc) {
    if (!sc->rendering) return RT_OK;
    CU(cudaSetDevice(sc->device));
    CU(cudaStreamSynchronize(sc->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, sc->ev_frame_start, sc->ev_frame_stop);
    sc->last_frame_ms = ms;
    resolve_spans(sc);
    sc->delivered = sc->batches.size();
    sc->rendering = false;
    sc->frame_complete = true;
    return RT_OK;
}

int rt_render_poll(rt_scene* sc, rt_vec3* buffer, int* done) {
    if (!sc || !done) return fail(RT_ERR_INVALID, "null argument");
    if (!sc->rendering) return fail(RT_ERR_STATE, "rt_render_poll without rt_render_start");
    if (sc->multi_active) return render_poll_multi(sc, buffer, done);
    CU(cudaSetDevice(sc->device));
    size_t ready = sc->delivered;
    while (ready < sc->batches.size()) {
        cudaError_t e = cudaEventQuery(sc->batches[ready].done);
        if (e == cudaSuccess) ready++;
        else if (e == cudaErrorNotReady) break;
        else return fail(RT_ERR_CUDA, std::string("render: ") + cudaGetErrorString(e));
    }
    if (ready > sc->delivered && buffer) {
        uint64_t q0 = sc->batches[sc->delivered].first_owned;
        uint64_t q1 = sc->batches[ready - 1].first_owned + sc->batches[ready - 1].n_pixels;
        int rc = deliver(sc, q0, q1, buffer);
        if (rc != RT_OK) return rc;
    }
    sc->delivered = ready;
    if (ready == sc->batches.size()) {
        cudaError_t e = cudaEventQuery(sc->ev_frame_stop);
        if (e == cudaErrorNotReady) {
            *done = 0;
            return RT_OK;
        }
        if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("render: ") + cudaGetErrorString(e));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, sc->ev_frame_start, sc->ev_frame_stop);
        sc->last_frame_ms = ms;
        resolve_spans(sc);
        if (sc->adaptive_frame) {   // paths = Σ counts: every pixel's pass-0 samples + the listed pixels' of every pass
            std::vector<uint32_t> live(sc->adaptive_m.size() - 1);
            if (!live.empty()) {
                CU(cudaMemcpyAsync(live.data(), sc->d_live, live.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, sc->copy_stream));
                CU(cudaStreamSynchronize(sc->copy_stream));
            }
            sc->paths += sc->owned_pixels * sc->adaptive_m[0];
            for (size_t k = 0; k < live.size(); k++) sc->paths += (uint64_t)live[k] * sc->adaptive_m[k + 1];
        }
        sc->rendering = false;
        sc->frame_complete = true;
        *done = 1;
        return RT_OK;
    }
    *done = 0;
    return RT_OK;
}

int rt_render_wait(rt_scene* sc, rt_vec3* buffer) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (!sc->rendering) return fail(RT_ERR_STATE, "rt_render_wait without rt_render_start");
    CU(cudaSetDevice(sc->device));
    if (sc->multi_active) CU(cudaEventSynchronize(sc->ev_multi_done));
    CU(cudaStreamSynchronize(sc->stream));
    int done = 0;
    int rc = rt_render_poll(sc, buffer, &done);
    if (rc != RT_OK) return rc;
    if (!done) return fail(RT_ERR_STATE, "frame did not complete");
    return RT_OK;
}

int rt_render_stop(rt_scene* sc) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (sc->multi_active)
        for (rt_scene* peer : sc->peers) rt_render_stop(peer);
    if (!sc->rendering) return RT_OK;
    cudaSetDevice(sc->device);
    // work already enqueued cannot be recalled; drain it so the buffers can be reused
    cudaStreamSynchronize(sc->stream);
    resolve_spans(sc);
    sc->rendering = false;
    sc->frame_complete = false;
    return RT_OK;
}

int rt_render_device_frame(rt_scene* sc, const rt_vec3** d_frame, uint64_t* n_pixels) {
    if (!sc || !d_frame || !n_pixels) return fail(RT_ERR_INVALID, "null argument");
    if (sc->rendering) {
        int rc = rt_render_wait(sc, nullptr);
        if (rc != RT_OK) return rc;
    }
    if (!sc->frame_complete) return fail(RT_ERR_STATE, "no completed frame");
    if (sc->multi_active) {
        *d_frame = sc->d_full_frame;
        *n_pixels = (uint64_t)sc->multi_rp.image.width * sc->multi_rp.image.height;
        return RT_OK;
    }
    if (sc->map.shard_count != 1) return fail(RT_ERR_STATE, "the last frame was one shard of a frame: use rt_render_device_result + rt_assemble_frame");
    *d_frame = sc->d_frame;   // owned order == x + y*width for an unsharded frame
    *n_pixels = (uint64_t)sc->map.width * sc->map.height;
    return RT_OK;
}

int rt_render_device_result(rt_scene* sc, const void** d_accum, uint64_t* n_float4) {
    if (!sc || !d_accum || !n_float4) return fail(RT_ERR_INVALID, "null argument");
    if (sc->multi_active) return fail(RT_ERR_STATE, "a multi-device handle delivers the assembled frame: rt_render_device_frame");
    if (sc->rendering) {
        CU(cudaSetDevice(sc->device));
        CU(cudaStreamSynchronize(sc->stream));
        int done = 0;
        int rc = rt_render_poll(sc, nullptr, &done);
        if (rc != RT_OK) return rc;
    }
    if (!sc->frame_complete) return fail(RT_ERR_STATE, "no completed frame");
    *d_accum = sc->d_accum;
    *n_float4 = sc->owned_pixels;
    return RT_OK;
}

uint64_t rt_shard_float4_count(const rt_render_params* p, uint32_t shard_index) {
    if (!p || p->image.width == 0 || p->image.height == 0) return 0;
    ShardMap m = make_shard_map(*p, shard_index);
    if (!tile_fits(m)) return 0;
    return owned_tiles(m) * m.tile_pixels();
}

int rt_assemble_frame(rt_scene* sc, const rt_render_params* p, const void* const* d_shards, rt_vec3* d_frame, void* stream) {
    if (!sc || !p || !d_shards || !d_frame) return fail(RT_ERR_INVALID, "null argument");
    uint32_t shard_count = p->shard_count ? p->shard_count : 1;
    if (shard_count > 16) return fail(RT_ERR_INVALID, "at most 16 shards");
    const uint64_t n_px = (uint64_t)p->image.width * p->image.height;
    if (n_px == 0 || n_px > 0xFFFFFFFFull) return fail(RT_ERR_INVALID, "empty or too large image");
    rt_render_params pp = *p;
    pp.shard_count = shard_count;
    ShardMap m = make_shard_map(pp, 0);
    if (!tile_fits(m)) return fail(RT_ERR_INVALID, "tile_width * tile_height >= 2^32");
    CU(cudaSetDevice(sc->device));
    ShardPtrs sp;
    for (uint32_t s = 0; s < 16; s++) sp.p[s] = s < shard_count ? (const Acc*)d_shards[s] : nullptr;
    cudaStream_t st = stream ? (cudaStream_t)stream : sc->stream;
    k_assemble<<<(unsigned)((n_px + 255) / 256), 256, 0, st>>>(sp, m, d_frame);
    sc->launches++;
    CU(cudaGetLastError());
    return RT_OK;
}

static int ensure_tone_out(rt_scene* sc, uint64_t n) {
    if (sc->tone_out_cap >= n) return RT_OK;
    cudaFree(sc->d_tone_out);
    sc->d_tone_out = nullptr;
    sc->tone_out_cap = 0;
    CU(cudaMalloc(&sc->d_tone_out, n * sizeof(uchar4)));
    sc->tone_out_cap = n;
    return RT_OK;
}

int rt_tonemap_rgba8(rt_scene* sc, const rt_vec3* frame, uint64_t n, uint8_t* rgba) {
    if (!sc || !frame || !rgba) return fail(RT_ERR_INVALID, "null argument");
    if (n == 0) return RT_OK;
    CU(cudaSetDevice(sc->device));
    if (sc->tone_in_cap < n) {   // persistent buffers, grown on demand: no allocation per call
        cudaFree(sc->d_tone_in);
        sc->d_tone_in = nullptr;
        sc->tone_in_cap = 0;
        CU(cudaMalloc(&sc->d_tone_in, n * sizeof(rt_vec3)));
        sc->tone_in_cap = n;
    }
    int rc = ensure_tone_out(sc, n);
    if (rc != RT_OK) return rc;
    CU(cudaMemcpyAsync(sc->d_tone_in, frame, n * sizeof(rt_vec3), cudaMemcpyHostToDevice, sc->copy_stream));
    k_tonemap<<<(unsigned)((n + 255) / 256), 256, 0, sc->copy_stream>>>(sc->d_tone_in, n, sc->d_tone_out);
    sc->launches++;
    CU(cudaMemcpyAsync(rgba, sc->d_tone_out, n * sizeof(uchar4), cudaMemcpyDeviceToHost, sc->copy_stream));
    cudaError_t e = cudaStreamSynchronize(sc->copy_stream);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("tonemap: ") + cudaGetErrorString(e));
    return RT_OK;
}

int rt_tonemap_rgba8_device(rt_scene* sc, const uint8_t** d_rgba, uint8_t* rgba_host, uint64_t* n_pixels) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    const rt_vec3* d_frame = nullptr;
    uint64_t n = 0;
    int rc = rt_render_device_frame(sc, &d_frame, &n);
    if (rc != RT_OK) return rc;
    CU(cudaSetDevice(sc->device));
    if ((rc = ensure_tone_out(sc, n)) != RT_OK) return rc;
    k_tonemap<<<(unsigned)((n + 255) / 256), 256, 0, sc->copy_stream>>>(d_frame, n, sc->d_tone_out);
    sc->launches++;
    if (rgba_host) CU(cudaMemcpyAsync(rgba_host, sc->d_tone_out, n * sizeof(uchar4), cudaMemcpyDeviceToHost, sc->copy_stream));
    cudaError_t e = cudaStreamSynchronize(sc->copy_stream);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("tonemap: ") + cudaGetErrorString(e));
    if (d_rgba) *d_rgba = reinterpret_cast<const uint8_t*>(sc->d_tone_out);
    if (n_pixels) *n_pixels = n;
    return RT_OK;
}

// ---- caller-supplied rays of many pixels (renderer::trace_pixel_samples_group, src/renderer/mod.rs:127-149) -------
static int check_groups(rt_scene* sc, const rt_ray* rays, uint64_t n_rays, const uint64_t* offsets,
                        const uint32_t* pixel_index, uint32_t n_groups, uint32_t max_depth, const rt_vec3* means) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (max_depth > RT_MAX_LEVELS - 2) return fail(RT_ERR_INVALID, "max_depth too large (limit 62)");
    if (n_groups == 0) return n_rays == 0 ? RT_OK : fail(RT_ERR_INVALID, "rays without groups");
    if (!offsets || !pixel_index || !means || (n_rays && !rays)) return fail(RT_ERR_INVALID, "null argument");
    if (offsets[0] != 0) return fail(RT_ERR_INVALID, "offsets[0] must be 0");
    for (uint32_t g = 0; g < n_groups; g++) {
        if (offsets[g + 1] < offsets[g]) return fail(RT_ERR_INVALID, "offsets decrease");
        if (offsets[g + 1] - offsets[g] > 0xFFFFFFFFull) return fail(RT_ERR_INVALID, "a group has 2^32 rays or more");
    }
    if (offsets[n_groups] != n_rays) return fail(RT_ERR_INVALID, "offsets[n_groups] must be n_rays");
    if (sc->rendering) return fail(RT_ERR_STATE, "a frame is in flight");
    return RT_OK;
}

struct GroupBatch {
    uint64_t r0, r1;   // rays [r0, r1) of the call
    uint32_t g0, g1;   // groups [g0, g1): every group with a ray in the batch (and the empty ones between them)
    int lane;
};

// Enqueue a validated call (n_groups > 0) on the library's streams; the main stream ends after every lane.  No host
// synchronisation.  Whole groups are packed in order into batches of at most RT_B200_BATCH_PATHS paths that alternate
// over the lanes like a frame's; a group larger than a batch is cut into batch-sized pieces that all run on ONE lane, so
// its running sum (k_group_resolve) passes from piece to piece in stream order and no lane reads another's partial sum.
static int trace_groups(rt_scene* sc, const rt_ray* d_rays, uint64_t n_rays, const uint64_t* offsets,
                        const uint32_t* pixel_index, uint32_t n_groups, uint32_t max_depth, uint64_t seed, rt_vec3* d_means) {
    uint64_t cap = std::min<uint64_t>(std::max<uint64_t>(env_size("RT_B200_BATCH_PATHS", (size_t)1 << 23), 1), 0xFFFFFFF0ull);
    int lanes_used = sc->ktiming ? 1 : sc->n_lanes;   // the lane policy of render_start_single
    if (!sc->lanes_from_env && lanes_used > 2 && (n_rays + cap - 1) / cap < 6) lanes_used = 2;
    if (lanes_used > 1) {
        const uint64_t split = (n_rays + lanes_used - 1) / lanes_used;
        if (split >= ((uint64_t)1 << 20)) cap = std::min(cap, split);
    }
    std::vector<GroupBatch> plan;
    uint64_t lane_paths[RT_MAX_LANES] = {0, 0, 0};
    uint64_t unit = 0;
    for (uint32_t g = 0; g < n_groups; unit++) {
        const int lane = (int)(unit % (uint64_t)lanes_used);
        const uint32_t g0 = g;
        const uint64_t r0 = offsets[g];
        if (offsets[g + 1] - r0 > cap) {
            for (uint64_t r = r0; r < offsets[g + 1]; r += cap)
                plan.push_back({r, std::min(r + cap, offsets[g + 1]), g, g + 1, lane});
            g++;
        } else {
            while (g < n_groups && offsets[g + 1] - r0 <= cap) g++;
            plan.push_back({r0, offsets[g], g0, g, lane});
        }
        lane_paths[lane] = std::max(lane_paths[lane], std::min<uint64_t>(offsets[g] - r0, cap));
    }
    lanes_used = (int)std::min<uint64_t>((uint64_t)lanes_used, unit);
    int rc = RT_OK;
    for (int l = 0; l < lanes_used && rc == RT_OK; l++) {
        bind_lane(sc, l);
        rc = ensure_path_buffers(sc, std::max<uint64_t>(lane_paths[l], 1024));
    }
    bind_lane(sc, 0);
    if (rc != RT_OK) return rc;
    if ((rc = ensure_device_array(sc->d_group_off, sc->group_off_cap, (uint64_t)n_groups + 1)) != RT_OK) return rc;
    if ((rc = ensure_device_array(sc->d_group_pix, sc->group_pix_cap, n_groups)) != RT_OK) return rc;
    auto enqueue = [&]() -> int {
        // the main stream is past the previous call (it waited for every lane) when it overwrites the offsets
        sc->h_group_off.assign(offsets, offsets + (uint64_t)n_groups + 1);
        sc->h_group_pix.assign(pixel_index, pixel_index + n_groups);
        CU(cudaMemcpyAsync(sc->d_group_off, sc->h_group_off.data(), ((uint64_t)n_groups + 1) * sizeof(uint64_t),
                           cudaMemcpyHostToDevice, sc->stream));
        CU(cudaMemcpyAsync(sc->d_group_pix, sc->h_group_pix.data(), (uint64_t)n_groups * sizeof(uint32_t),
                           cudaMemcpyHostToDevice, sc->stream));
        CU(cudaEventRecord(sc->ev_group_start, sc->stream));
        for (int l = 1; l < lanes_used; l++) CU(cudaStreamWaitEvent(sc->lanes[l].stream, sc->ev_group_start, 0));
        for (const GroupBatch& b : plan) {
            bind_lane(sc, b.lane);
            const uint32_t n = (uint32_t)(b.r1 - b.r0), ng = b.g1 - b.g0;
            if (n > 0) {
                CU(cudaMemsetAsync(sc->d_counts, 0, RT_CNT_WORDS * sizeof(uint32_t), sc->stream));
                {
                    KernelSpan span(sc, RT_KCLASS_RAYGEN);
                    k_load_groups<<<(unsigned)(((uint64_t)n + 255) / 256), 256, 0, sc->stream>>>(
                        d_rays + b.r0, n, b.r0, sc->d_group_off + b.g0, sc->d_group_pix + b.g0, ng, sc->q[0], sc->d_counts, sc->hq.key);
                }
                launch_bounces(sc, max_depth, seed);
            }
            {
                KernelSpan span(sc, RT_KCLASS_RESOLVE);
                k_group_resolve<<<(unsigned)(((uint64_t)ng + 255) / 256), 256, 0, sc->stream>>>(
                    sc->d_radiance, b.r0, b.r1, sc->d_group_off + b.g0, ng, d_means + b.g0);
            }
        }
        bind_lane(sc, 0);
        for (int l = 1; l < lanes_used; l++) {
            CU(cudaEventRecord(sc->lanes[l].done, sc->lanes[l].stream));
            CU(cudaStreamWaitEvent(sc->stream, sc->lanes[l].done, 0));
        }
        CU(cudaGetLastError());
        return RT_OK;
    };
    rc = enqueue();
    bind_lane(sc, 0);
    if (rc != RT_OK) return rc;
    sc->paths += n_rays;
    return RT_OK;
}

int rt_trace_pixel_samples_group_device(rt_scene* sc, const rt_ray* d_rays, uint64_t n_rays, const uint64_t* offsets,
                                        const uint32_t* pixel_index, uint32_t n_groups, uint32_t max_depth, uint64_t seed,
                                        rt_vec3* d_means, void* stream) {
    int rc = check_groups(sc, d_rays, n_rays, offsets, pixel_index, n_groups, max_depth, d_means);
    if (rc != RT_OK || n_groups == 0) return rc;
    CU(cudaSetDevice(sc->device));
    cudaStream_t caller = (cudaStream_t)stream;   // NULL: the library's stream
    if (caller) {
        CU(cudaEventRecord(sc->ev_group_in, caller));
        CU(cudaStreamWaitEvent(sc->stream, sc->ev_group_in, 0));
    }
    if ((rc = trace_groups(sc, d_rays, n_rays, offsets, pixel_index, n_groups, max_depth, seed, d_means)) != RT_OK) return rc;
    if (caller) {   // work the caller queues next (e.g. freeing the rays) runs after the last read of d_rays / write of d_means
        CU(cudaEventRecord(sc->ev_group_done, sc->stream));
        CU(cudaStreamWaitEvent(caller, sc->ev_group_done, 0));
    }
    if (sc->ktiming) {   // the event pairs of the kernel timing are read once the work has run
        CU(cudaStreamSynchronize(sc->stream));
        resolve_spans(sc);
    }
    return RT_OK;
}

int rt_trace_pixel_samples_group(rt_scene* sc, const rt_ray* rays, uint64_t n_rays, const uint64_t* offsets,
                                 const uint32_t* pixel_index, uint32_t n_groups, uint32_t max_depth, uint64_t seed,
                                 rt_vec3* means) {
    int rc = check_groups(sc, rays, n_rays, offsets, pixel_index, n_groups, max_depth, means);
    if (rc != RT_OK || n_groups == 0) return rc;
    CU(cudaSetDevice(sc->device));
    if ((rc = ensure_device_array(sc->d_group_rays, sc->group_rays_cap, n_rays)) != RT_OK) return rc;
    if ((rc = ensure_device_array(sc->d_group_means, sc->group_means_cap, n_groups)) != RT_OK) return rc;
    if (n_rays) CU(cudaMemcpyAsync(sc->d_group_rays, rays, n_rays * sizeof(rt_ray), cudaMemcpyHostToDevice, sc->stream));
    if ((rc = trace_groups(sc, sc->d_group_rays, n_rays, offsets, pixel_index, n_groups, max_depth, seed, sc->d_group_means)) != RT_OK)
        return rc;
    CU(cudaMemcpyAsync(means, sc->d_group_means, (uint64_t)n_groups * sizeof(rt_vec3), cudaMemcpyDeviceToHost, sc->stream));
    const cudaError_t e = cudaStreamSynchronize(sc->stream);
    resolve_spans(sc);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("trace_pixel_samples_group: ") + cudaGetErrorString(e));
    return RT_OK;
}

// the one-group case
int rt_trace_pixel_samples(rt_scene* sc, const rt_ray* rays, uint32_t n_rays, uint32_t max_depth, uint64_t seed,
                           uint32_t pixel_index, rt_vec3* mean_out) {
    if (!sc || !rays || !mean_out) return fail(RT_ERR_INVALID, "null argument");
    if (n_rays == 0) return fail(RT_ERR_INVALID, "no rays");
    const uint64_t offsets[2] = {0, n_rays};
    return rt_trace_pixel_samples_group(sc, rays, n_rays, offsets, &pixel_index, 1, max_depth, seed, mean_out);
}

// ---- instrumentation ---------------------------------------------------------------------------
int rt_get_stats(rt_scene* sc, rt_stats* out) {
    if (!sc || !out) return fail(RT_ERR_INVALID, "null argument");
    CU(cudaSetDevice(sc->device));
    DevCounters c;
    CU(cudaMemcpy(&c, sc->d_counters, sizeof c, cudaMemcpyDeviceToHost));
    out->kernel_launches = sc->launches;
    out->paths = sc->paths;
    out->segments = c.segments;
    out->shape_tests = c.shape_tests;
    out->cull_tests = c.cull_tests;
    out->march_steps = c.march_steps;
    out->march_rays = c.march_rays;
    out->march_long_rays = c.march_long_rays;
    out->march_max_evals = c.march_max_evals;
    out->last_frame_ms = sc->last_frame_ms;
    out->last_intersect_ms = sc->last_intersect_ms;
    out->verify_rays = c.verify_rays;
    out->verify_false_culls = c.verify_false_culls;
    for (int k = 0; k < 8; k++) out->march_prof[k] = c.march_prof[k];
    out->ms_raygen = sc->ms_cls[RT_KCLASS_RAYGEN];
    out->ms_extend = sc->ms_cls[RT_KCLASS_EXTEND];
    out->ms_march = sc->ms_cls[RT_KCLASS_MARCH];
    out->ms_shade = sc->ms_cls[RT_KCLASS_SHADE];
    out->ms_resolve = sc->ms_cls[RT_KCLASS_RESOLVE];
    out->launches_extend = sc->n_cls[RT_KCLASS_EXTEND];
    out->launches_march = sc->n_cls[RT_KCLASS_MARCH];
    out->launches_shade = sc->n_cls[RT_KCLASS_SHADE];
    return RT_OK;
}
int rt_reset_stats(rt_scene* sc) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    CU(cudaSetDevice(sc->device));
    CU(cudaMemset(sc->d_counters, 0, sizeof(DevCounters)));
    sc->launches = 0;
    sc->paths = 0;
    for (int k = 0; k < RT_KCLASS_COUNT; k++) { sc->ms_cls[k] = 0.0; sc->n_cls[k] = 0; }
    return RT_OK;
}
int rt_set_counters(rt_scene* sc, int enabled) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    sc->counters_on = enabled != 0;
    return RT_OK;
}
int rt_set_kernel_timing(rt_scene* sc, int enabled) {
    if (!sc) return fail(RT_ERR_INVALID, "null scene");
    if (sc->rendering) return fail(RT_ERR_STATE, "a frame is in flight");
    sc->ktiming = enabled != 0;
    return RT_OK;
}

int rt_march_region_bounds(const double* params8, double* grad_bound, double* hess_bound) {
    if (!params8 || !grad_bound || !hess_bound) return fail(RT_ERR_INVALID, "null argument");
    if (!(params8[0] >= 0 && params8[0] <= RT_SURF_CUSHION)) return fail(RT_ERR_INVALID, "unknown surface kind");
    bounds::region_bounds(params8, grad_bound, hess_bound);
    return RT_OK;
}

int rt_advance_exact(double a, double s, int64_t m, double* out) {
    if (!out) return fail(RT_ERR_INVALID, "null argument");
    *out = advance_exact(a, s, (long long)m);
    return RT_OK;
}

int rt_div3_exact(const double* a, const double* s, uint64_t n, double* q) {
    if (!a || !s || !q) return fail(RT_ERR_INVALID, "null argument");
    for (uint64_t i = 0; i < n; i++) div3_exact(a[3 * i], a[3 * i + 1], a[3 * i + 2], s[i], q[3 * i], q[3 * i + 1], q[3 * i + 2]);
    return RT_OK;
}

int rt_march_candidates_host(const double* params8, const double* inverse12, const rt_ray* rays, uint64_t n, double t_min,
                             double t_max, double best, int miss_proof, double* t_out, uint8_t* hit_out, uint64_t* evaluations) {
    if (!params8 || !inverse12 || (n && !rays) || !t_out || !hit_out) return fail(RT_ERR_INVALID, "null argument");
    const int kind = (int)params8[0];
    if (!(kind >= RT_SURF_HEART && kind <= RT_SURF_CUSHION)) return fail(RT_ERR_INVALID, "unknown surface kind");
    double G, H;
    bounds::region_bounds(params8, &G, &H);
    const double F = bounds::region_magnitude(params8);
    unsigned long long total = 0;
    for (uint64_t i = 0; i < n; i++) {
        const D3 ro = mk(rays[i].origin.x, rays[i].origin.y, rays[i].origin.z);
        const D3 rd = mk(rays[i].direction.x, rays[i].direction.y, rays[i].direction.z);
        // march_needed (rt_scene.cuh), host side: object-space ray, bounding chord, clipped by the best hit so far
        const D3 o = xf_point(inverse12, ro), d = xf_vector(inverse12, rd);
        double start, end, t = 0.0;
        bool hit = false;
        if (march_bound(params8, o, d, start, end)) {
            double end_c = end;
            bool needed = true;
            if (params8[1] > 0.0) {
                if (!(start <= best)) needed = false;
                end_c = fmin(end, best + 2.0 * params8[1]);
            }
            if (needed) {
                unsigned long long ev = 0;
                hit = march_candidate_skip(params8, o, d, start, end_c, t_min, t_max, G, F, t, ev, miss_proof != 0);
                total += ev;
            }
        }
        hit_out[i] = hit ? 1 : 0;
        t_out[i] = hit ? t : 0.0;
    }
    if (evaluations) *evaluations = total;
    return RT_OK;
}

int rt_bernstein_clear(const double* coefficients, int degree, double length, double threshold, int* clear) {
    if (!coefficients || !clear) return fail(RT_ERR_INVALID, "null argument");
    if (degree == 6) {
        double c[7];
        for (int k = 0; k <= 6; k++) c[k] = coefficients[k];
        *clear = bernstein_clear<6>(c, length, threshold) ? 1 : 0;
    } else if (degree == 4) {
        double c[5];
        for (int k = 0; k <= 4; k++) c[k] = coefficients[k];
        *clear = bernstein_clear<4>(c, length, threshold) ? 1 : 0;
    } else {
        return fail(RT_ERR_INVALID, "degree must be 4 or 6 (the marched surfaces' degrees along a ray)");
    }
    return RT_OK;
}

int rt_cull_tree_check(const rt_scene_desc* d, uint32_t* n_roots, uint32_t* n_groups, uint32_t* n_tree,
                       uint32_t* n_flat, double* worst) {
    int rc = validate_desc(d);
    if (rc != RT_OK) return rc;
    if (!n_roots || !n_groups || !n_tree || !n_flat || !worst) return fail(RT_ERR_INVALID, "null argument");
    const int n = (int)d->n_shapes;
    CullTree ct = cull_build(d->inverse, d->kind, n, false, false, d->params);
    *n_roots = (uint32_t)ct.n_roots;
    *n_groups = (uint32_t)ct.n_groups;
    *n_flat = (uint32_t)ct.n_flat_real;
    const float4* roots = ct.table.data();
    const float4* grp = roots + ct.n_roots;
    // radius a node entry stands for: A = 1.0101 (s R + sqrt(3B)(|c| + R))^2  ->  R
    auto node_radius = [](float4 e) {
        const double cn = sqrt((double)e.x * e.x + (double)e.y * e.y + (double)e.z * e.z);
        const double x = sqrt((double)e.w / 1.0101);
        return (x - sqrt(3.0 * RT_CULL_B) * cn) / (sqrt(1.1) + sqrt(3.0 * RT_CULL_B));
    };
    double w = -INFINITY;
    uint32_t in_tree = 0;
    std::vector<double> group_reach_c(3 * (size_t)ct.n_groups, 0.0), group_r((size_t)ct.n_groups, -1.0);
    for (int i = 0; i < n; i++) {
        const int g = ct.group_of[i];
        if (g < 0) continue;
        in_tree++;
        if (g >= ct.n_groups || !isfinite(grp[g].w)) return fail(RT_ERR_STATE, "cull tree: shape in a padding group");
        // the shape's true world ball, from its own transform (not from the table entry)
        double r;
        const double* qi = d->params + (size_t)RT_SHAPE_PARAMS * i;
        const float4 leaf = cull_entry(d->inverse + (size_t)12 * i, d->kind[i], &r, fabs(qi[0]) + fabs(qi[1]));
        const double* m = d->direct + (size_t)12 * i;   // centre = direct * origin
        const double c[3] = {m[3], m[7], m[11]};
        (void)leaf;
        const double gr = node_radius(grp[g]);
        const double dx = c[0] - grp[g].x, dy = c[1] - grp[g].y, dz = c[2] - grp[g].z;
        w = fmax(w, (sqrt(dx * dx + dy * dy + dz * dz) + r - gr) / gr);
        group_r[g] = gr;
        const float4 rt_ = roots[g / RT_CULL_ROOT_FANOUT];
        const double rr = node_radius(rt_);
        const double ex = grp[g].x - rt_.x, ey = grp[g].y - rt_.y, ez = grp[g].z - rt_.z;
        w = fmax(w, (sqrt(ex * ex + ey * ey + ez * ez) + ct.group_radius[g] - rr) / rr);
        // and the leaf directly under the root
        const double fx = c[0] - rt_.x, fy = c[1] - rt_.y, fz = c[2] - rt_.z;
        w = fmax(w, (sqrt(fx * fx + fy * fy + fz * fz) + r - rr) / rr);
    }
    // levels above the roots: every node encloses the nodes it covers (FP64 balls of the build)
    {
        std::vector<CullBall> below = ct.root_ball;
        size_t at = 0;
        for (int l = 1; l <= ct.n_upper; l++) {
            std::vector<CullBall> here(ct.upper_ball.begin() + at, ct.upper_ball.begin() + at + ct.upper_count[l]);
            at += ct.upper_count[l];
            for (int i = 0; i < ct.upper_count[l]; i++) {
                const double nr = node_radius(ct.upper[ct.upper_off[l] + i]);
                for (int k = 32 * i; k < std::min(32 * i + 32, (int)below.size()); k++) {
                    if (below[k].r < 0.0) continue;
                    const double dx = below[k].c[0] - here[i].c[0], dy = below[k].c[1] - here[i].c[1], dz = below[k].c[2] - here[i].c[2];
                    w = fmax(w, (sqrt(dx * dx + dy * dy + dz * dz) + below[k].r - nr) / nr);
                }
            }
            below = here;
        }
    }
    *n_tree = in_tree;
    *worst = in_tree ? w : 0.0;
    return RT_OK;
}

int rt_cull_reached(const rt_scene_desc* d, const rt_ray* rays, uint64_t n_rays, uint8_t* reached) {
    int rc = validate_desc(d);
    if (rc != RT_OK) return rc;
    if ((n_rays && !rays) || !reached) return fail(RT_ERR_INVALID, "null argument");
    const int n = (int)d->n_shapes;
    const CullTree ct = cull_build(d->inverse, d->kind, n, false, false, d->params);
    std::vector<std::pair<int, float4>> march;  // (shape, ball around its marching bound), like rt_scene_create
    for (int i = 0; i < n; i++) {
        if (d->kind[i] != RT_SHAPE_MARCH) continue;
        const double* q = d->params + (size_t)i * RT_SHAPE_PARAMS;
        double radius[3] = {q[7], q[7], q[7]};
        if ((int)q[0] == RT_SURF_HEART) { radius[0] = 1.45; radius[1] = 1.45 / 2.05; radius[2] = 1.45; }
        march.push_back({i, cull_entry_march_bound(d->inverse + (size_t)12 * i, radius)});
    }
    const float4* roots = ct.table.data();
    const float4* groups = roots + ct.n_roots;
    const float4* leaves = groups + ct.n_groups;
    const float4* flat = leaves + (size_t)RT_CULL_GROUP * ct.n_groups;
    const int* leaf_ids = ct.ids.data();
    const int* flat_ids = leaf_ids + (size_t)RT_CULL_GROUP * ct.n_groups;
    for (uint64_t r = 0; r < n_rays; r++) {
        uint8_t* out = reached + r * (uint64_t)n;
        memset(out, 0, (size_t)n);
        const rt_ray& ray = rays[r];
        const CullRay cr = make_cull_ray(ray.origin.x, ray.origin.y, ray.origin.z, ray.direction.x, ray.direction.y,
                                         ray.direction.z);
        for (int j = 0; j < ct.n_flat; j++)
            if (flat_ids[j] >= 0 && cull_pass(cr, flat[j])) out[flat_ids[j]] = 1;
        for (int rt_i = 0; rt_i < ct.n_roots; rt_i++) {
            bool above = true;   // the upper levels (the device skips a rejected node's whole range: same decisions)
            for (int l = 1; l <= ct.n_upper && above; l++)
                above = cull_pass_node(cr, ct.upper[ct.upper_off[l] + (rt_i >> (5 * l))]);
            if (!above) continue;
            if (!cull_pass_node(cr, roots[rt_i])) continue;
            const int g0 = RT_CULL_ROOT_FANOUT * rt_i, g1 = std::min(g0 + RT_CULL_ROOT_FANOUT, ct.n_groups);
            for (int g = g0; g < g1; g++) {
                if (!cull_pass_node(cr, groups[g])) continue;
                for (int j = 0; j < RT_CULL_GROUP; j++) {
                    const int id = leaf_ids[(size_t)RT_CULL_GROUP * g + j];
                    if (id >= 0 && cull_pass(cr, leaves[(size_t)RT_CULL_GROUP * g + j])) out[id] = 1;
                }
            }
        }
        for (auto& m : march)
            if (cull_pass(cr, m.second)) out[m.first] = 1;
    }
    return RT_OK;
}

int rt_measure_peaks(int device, double* fp64_tflops, double* fp32_tflops) {
    int ndev = rt_device_count();
    if (ndev == 0) return fail(RT_ERR_NO_DEVICE, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(RT_ERR_INVALID, "device index out of range");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    void* buf = nullptr;
    CU(cudaMalloc(&buf, (size_t)blocks * threads * sizeof(double)));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    auto run = [&](bool dbl, int iters) -> double {
        float best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {
            cudaEventRecord(a);
            if (dbl) k_fma_peak<double><<<blocks, threads>>>((double*)buf, iters, 1.0000001, 1e-9);
            else k_fma_peak<float><<<blocks, threads>>>((float*)buf, iters, 1.0000001f, 1e-9f);
            cudaEventRecord(b);
            cudaEventSynchronize(b);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, a, b);
            if (rep > 0 && ms < best) best = ms;
        }
        double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
        return flops / (best * 1e-3) / 1e12;
    };
    if (fp64_tflops) *fp64_tflops = run(true, 1 << 14);
    if (fp32_tflops) *fp32_tflops = run(false, 1 << 15);
    cudaError_t e = cudaDeviceSynchronize();
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(buf);
    if (e != cudaSuccess) return fail(RT_ERR_CUDA, std::string("measure_peaks: ") + cudaGetErrorString(e));
    return RT_OK;
}

}  // extern "C"
