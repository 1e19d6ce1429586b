// Path-state queues of the wavefront renderer and the helpers shared by its translation units
// (rt_core.cu: raygen / extend / shade / resolve + the C ABI; rt_march3.cu: the pooled marching kernel).
#pragma once
#include "rt_scene.cuh"

using namespace rt;

#define RT_MAX_LEVELS 64  // counters per batch: level 0 .. max_depth + 1

// ------------------------------------------------------------------------------------------------
// path state: structure of arrays in HBM, two queues (ping-pong per bounce)
// ------------------------------------------------------------------------------------------------
struct PathQueue {
    double *ox, *oy, *oz, *dx, *dy, *dz;  // ray
    double *bx, *by, *bz;                 // throughput (product of attenuations so far)
    uint32_t* pid;                        // path id inside the batch = pixel_local * spp + sample
};

struct HitQueue {
    double* t;        // best t so far (max_t = +inf when nothing was hit)
    int32_t* index;   // winning shape, -1 = none
    uint32_t* mq_slot;  // march queue: path slot ...
    uint32_t* mq_mask;  // ... and the marched shapes (bit k = S.march_index[k]) it still has to test
    uint32_t* fq_slot;  // the march queue after k_march_filter: the entries that still have a shape to march, compacted
    uint32_t* fq_mask;
    uint32_t* rq_slot;  // replay queue: degenerate rays (Sphere D == 0, NaN t) that must go through the literal loop
    uint2* key;         // [path id] the path's RNG key (image pixel index, sample), written once by k_extend's raygen,
                        // k_raygen or k_load_groups: k_shade / k_bounce read 8 B instead of redoing six integer divisions
                        // per segment, and caller-supplied rays need no pixel geometry at all
};

// per-level counters of one batch (zeroed by one memset): live paths, march / replay queue lengths and
// the march kernels' queue heads (one per surface kind)
#define RT_CNT_LIVE 0
#define RT_CNT_MARCH (RT_MAX_LEVELS)
#define RT_CNT_REPLAY (2 * RT_MAX_LEVELS)
#define RT_CNT_HEAD (3 * RT_MAX_LEVELS)              // + kind * RT_MAX_LEVELS
#define RT_CNT_FILTERED (9 * RT_MAX_LEVELS)          // length of the filtered march queue
#define RT_CNT_WORDS (10 * RT_MAX_LEVELS)

// append to a queue: one atomic per warp (ballot + popc); must be called by all 32 lanes of a warp
__device__ __forceinline__ uint32_t queue_append(bool alive, uint32_t* counter) {
    unsigned mask = __ballot_sync(0xffffffffu, alive);
    if (mask == 0) return 0;
    int lane = threadIdx.x & 31;
    int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(mask & ((1u << lane) - 1u));
}

__device__ __forceinline__ void flush_counters(const DevCounters& c, DevCounters* g) {
    // warp-reduce, one atomic per warp and counter
    unsigned long long v[6] = {c.segments, c.shape_tests, c.cull_tests, c.march_steps, c.march_rays, c.march_long_rays};
    unsigned long long mx = c.march_max_evals;
    for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_down_sync(0xffffffffu, mx, o));
#pragma unroll
    for (int k = 0; k < 6; k++) {
        unsigned long long x = v[k];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        v[k] = x;
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&g->segments, v[0]);
        atomicAdd(&g->shape_tests, v[1]);
        atomicAdd(&g->cull_tests, v[2]);
        atomicAdd(&g->march_steps, v[3]);
        atomicAdd(&g->march_rays, v[4]);
        atomicAdd(&g->march_long_rays, v[5]);
        atomicMax(&g->march_max_evals, mx);
    }
    if (c.verify_rays) atomicAdd(&g->verify_rays, c.verify_rays);
    if (c.verify_false_culls) atomicAdd(&g->verify_false_culls, c.verify_false_culls);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        unsigned long long x = c.march_prof[k];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(&g->march_prof[k], x);
    }
}

// a marched candidate came out NaN: the sequential loop is not an arg-min for this ray -> literal loop
static __device__ __noinline__ void replay_brute(const DevScene& S, const PathQueue& in, const HitQueue& hq, uint32_t i) {
    D3 ro = mk(in.ox[i], in.oy[i], in.oz[i]);
    D3 rd = mk(in.dx[i], in.dy[i], in.dz[i]);
    double best;
    int winner;
    DevCounters cc = {};
    nearest_hit_brute<false>(S, ro, rd, 0.001, INFINITY, best, winner, cc);
    hq.t[i] = best;
    hq.index[i] = winner;
}


// ---- the marching kernels live in their own translation units (rt_march_kernels.cu: k_march, k_march2;
//      rt_march3.cu: k_march3); rt_core.cu launches them through this interface -----------------------------
struct MarchLaunch {
    DevScene ds;
    int kind;                 // surface kind of this pass (one launch per kind present in the scene)
    uint32_t kind_mask;       // bits of the march-queue mask that belong to it
    PathQueue in;
    HitQueue hq;
    const uint32_t* march_count;
    uint32_t* head;
    DevCounters* counters;
    bool count;
    cudaStream_t stream;
    int version;              // 1 k_march, 2 k_march2, 3 k_march3
    int grid1, grid2, grid3;
    size_t smem3;
    int3 tune;
    void* march_state;        // k_march2's records
    bool prefiltered;         // k_march_filter has run on this queue: k_march need not try the hull proof again
    int grid_filter;
    uint32_t* filtered_count; // k_march_filter: length of the compacted queue it writes (hq.fq_slot / fq_mask)
};
void rt_launch_march(const MarchLaunch& ml);
void rt_launch_march_filter(const MarchLaunch& ml);   // once per level, before the per-kind launches
void rt_launch_march3(const MarchLaunch& ml);
// CTAs per SM of k_march / k_march2 / k_march3 and k_march3's dynamic shared memory per CTA
void rt_march_occupancy(int per_sm[3], size_t* smem3);
int rt_march3_occupancy(size_t* smem3);
size_t rt_march2_state_bytes(int grid2);
