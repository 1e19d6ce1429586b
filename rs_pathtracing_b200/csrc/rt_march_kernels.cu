// rt_march_kernels.cu -- K3 of the wavefront renderer: the miss proof for every queued (ray, marched shape) pair
// with full warps (k_march_filter), then exact-skip marching of what it leaves with ONE RAY PER LANE (k_march:
// persistent lanes, phase voting, cooperative exact advance), one launch per surface kind.  Compile with
// -fmad=false (see rt_math.cuh).
#include <cuda_runtime.h>
#include <cstdio>

#include <algorithm>

#include "rt_queues.cuh"

// The exact advance of a jump (rt_march.cuh, advance_exact) for every jumping lane of the warp: 4 tasks
// per lane (t, p.x, p.y, p.z), dealt out one per lane, so that the loops over binades -- whose trip
// counts differ wildly between accumulators -- run with up to 32 lanes busy instead of one lane doing its
// four advances in a row while the others wait.  Must be called by the whole warp (convergent).
template <class CoWork>
__device__ __forceinline__ void coop_advance(unsigned jumping, long long mj, double t, double step, D3 p, D3 sd,
                                             double& nt, D3& np, unsigned char* s_owner, CoWork&& co_work) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int tasks = 4 * __popc(jumping);
    const int my_rank = __popc(jumping & ((1u << lane) - 1u));
    const int my_first = 4 * my_rank;  // task number of this lane's t
    // the lane that owns task number k is the (k / 4)-th set bit of `jumping`: every jumping lane posts its
    // number at its rank (s_owner: 32 bytes of shared memory private to the warp; __fns is a long software
    // loop, stripping the lower bits one by one was 3.7 % of k_march's instructions)
    __syncwarp();
    if ((jumping >> lane) & 1u) s_owner[my_rank] = (unsigned char)lane;
    __syncwarp();
    double out[4] = {0.0, 0.0, 0.0, 0.0};
    for (int base = 0; base < tasks; base += 32) {
        const int task = base + lane;
        const bool active = task < tasks;
        const int src = active ? (int)s_owner[task >> 2] : lane;
        const int comp = task & 3;
        const double a0 = __shfl_sync(FULL, t, src), a1 = __shfl_sync(FULL, p.x, src), a2 = __shfl_sync(FULL, p.y, src),
                     a3 = __shfl_sync(FULL, p.z, src);
        const double s0 = __shfl_sync(FULL, step, src), s1 = __shfl_sync(FULL, sd.x, src),
                     s2 = __shfl_sync(FULL, sd.y, src), s3 = __shfl_sync(FULL, sd.z, src);
        const long long mm = __shfl_sync(FULL, mj, src);
        double res = comp == 0 ? a0 : comp == 1 ? a1 : comp == 2 ? a2 : a3;
        const double s = comp == 0 ? s0 : comp == 1 ? s1 : comp == 2 ? s2 : s3;
        long long left = active ? mm : 0;
        // one binade (or one stretch of the near-zero walk) per trip; the lanes whose task is finished -- or
        // that never had one -- do their co-work (literal steps of their own rays) instead of idling
#ifdef RT_MARCH_WATCHDOG
        unsigned long long wd_adv = 0;
#endif
        while (__any_sync(FULL, left > 0)) {
            if (left > 0) advance_iter(res, s, left);
            co_work();
#ifdef RT_MARCH_WATCHDOG
            if (++wd_adv == 5000000ull) {
                if (RT_MARCH_WATCHDOG == 1) printf("WD-ADV blk %d lane %d: left %lld res %.17g s %.17g mm %lld comp %d\n", blockIdx.x, threadIdx.x, left, res, s, mm, comp);
                left = 0;
            }
#endif
        }
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int from = my_first + c - base;  // lane holding this lane's result number c in this round
            const double v = __shfl_sync(FULL, res, from & 31);
            if (from >= 0 && from < 32) out[c] = v;
        }
    }
    nt = out[0];
    np = mk(out[1], out[2], out[3]);
}

// K3: exact-skip marching of the queued (ray, marched shapes) entries, one surface kind per launch.
// Per-ray cost is heavy-tailed (a grazing ray needs 50x the work of a typical one), so lanes are
// persistent: a lane that finishes its entry takes the next one from the queue (warp-aggregated atomic on
// `head`) while the other lanes of its warp keep marching.
#ifndef RT_MARCH_MIN_BLOCKS
#define RT_MARCH_MIN_BLOCKS 4
#endif
// tune.x: refill / start a shape when at least this many lanes of the warp are idle (or none is busy)
// tune.y: run the attempt phase when this many lanes want it (or nobody can step)
// tune.z: literal steps per literal phase
#define RT_MARCH_REFILL_MIN tune.x
#define RT_MARCH_ATTEMPT_MIN tune.y
#define RT_MARCH_LITERAL_BURST tune.z
template <int KIND, bool COUNT>
__global__ void __launch_bounds__(128, RT_MARCH_MIN_BLOCKS)
k_march(DevScene S, uint32_t kind_mask, PathQueue in, HitQueue hq, const uint32_t* __restrict__ march_count,
        uint32_t* head, DevCounters* g_counters, int3 tune) {
    DevCounters c = {};
    const uint32_t n = *march_count;
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    __shared__ unsigned char s_owner_all[128];
    unsigned char* const s_owner = s_owner_all + (threadIdx.x & ~31u);
    bool have = false, marching = false, exhausted = false;
    uint32_t slot = 0, mask = 0, entry = 0;
    int shape = -1, winner = -1;
    double best = 0.0;
    Marcher<KIND, COUNT> m;
    // the shape a lane marched is over (phase() == RT_PHASE_END): take its candidate
    auto finish_shape = [&]() {
        marching = false;
        if (COUNT) {
            c.march_steps += m.n;
            for (int k = 0; k < 8; k++) c.march_prof[k] += m.prof[k];
            if (m.n > 2048) c.march_long_rays++;
            if (m.n > c.march_max_evals) c.march_max_evals = m.n;
        }
        if (m.finish() == RT_MARCH_DONE && !(m.t < 0.001)) {  // ray_marching.rs:55 with max_t = +inf
            const double t = m.t;
            if (t != t) {  // NaN candidate: replay now, and hide the entry from later kind passes
                replay_brute(S, in, hq, slot);
                hq.mq_mask[entry] = 0;
                have = false;
            } else if (t < best || (t == best && shape > winner)) {
                best = t;
                winner = shape;
            }
        }
    };
#ifdef RT_MARCH_WATCHDOG
    unsigned long long wd_iter = 0;
#endif
    for (;;) {
#ifdef RT_MARCH_WATCHDOG
        if (++wd_iter == 20000000ull || wd_iter == 20000001ull) {
            if (RT_MARCH_WATCHDOG == 2 && lane == 0) atomicAdd(&g_counters->verify_rays, 1ull);
            if (RT_MARCH_WATCHDOG == 1) printf("WD blk %d lane %d it %llu: have %d marching %d exh %d mask %x entry %u slot %u | ph %d it %d depth %d t %.17g start %.17g end %.17g step %.17g r %.6g cooldown %d backoff %d skip_ok %d n %llu\n",
                   blockIdx.x, threadIdx.x, wd_iter, (int)have, (int)marching, (int)exhausted, mask, entry, slot,
                   marching ? m.phase() : -1, m.it, m.depth, m.t, m.start, m.end, m.step, m.r, m.cooldown, m.backoff, (int)m.skip_ok, m.n);
            if (wd_iter == 20000001ull) break;
        }
#endif
        // ---- fill: lanes without a ray in flight fetch queue entries and start their shapes, again and again
        //      (the `continue` below), until (nearly) every lane holds a ray that really has to be marched.  Entries
        //      whose chord the best hit now clips away (march_needed: an earlier kind pass may have lowered it since
        //      k_march_filter ran) never get that far, so what is left in the lanes is the expensive minority.  (No
        //      hull proof in begin(): k_march_filter has tried it for every entry of this queue.)
        //      (Written as part of the one outer loop on purpose: the same logic as a nested `for (;;)` with two
        //      breaks hung k_march<Cushion> / k_march<Dupin> on the second frame of a scene -- deterministically per
        //      binary, gone with any instrumentation; profiles/README.md, r2n.  Keep the nesting shallow.) ---------
        {
            const unsigned need = __ballot_sync(FULL, !marching && !exhausted);
            const unsigned marching_any = __ballot_sync(FULL, marching);
            if (need != 0 && (marching_any == 0 || __popc(need) >= RT_MARCH_REFILL_MIN)) {
                if (have && !marching && mask == 0) {   // every shape of the entry is done
                    hq.t[slot] = best;
                    hq.index[slot] = winner;
                    have = false;
                }
                const unsigned idle = __ballot_sync(FULL, !have && !exhausted);
                if (idle) {
                    uint32_t base = 0;
                    const int leader = __ffs(idle) - 1;
                    if (lane == leader) base = atomicAdd(head, (uint32_t)__popc(idle));
                    base = __shfl_sync(FULL, base, leader);
                    if (!have && !exhausted) {
                        const uint32_t j = base + __popc(idle & ((1u << lane) - 1u));
                        if (j < n) {
                            entry = j;
                            slot = hq.mq_slot[j];
                            mask = hq.mq_mask[j] & kind_mask;
                            best = hq.t[slot];
                            winner = hq.index[slot];
                            have = mask != 0;
                        } else {
                            exhausted = true;
                        }
                    }
                }
                if (have && !marching && mask != 0) {   // the entry's next marched shape
                    const int k = __ffs(mask) - 1;
                    mask &= mask - 1;
                    shape = S.march_index[k];
                    const double* q = S.params + RT_SHAPE_PARAMS * shape;
                    D3 ro = mk(in.ox[slot], in.oy[slot], in.oz[slot]);
                    D3 rd = mk(in.dx[slot], in.dy[slot], in.dz[slot]);
                    D3 o, d;
                    double start, end_c;
                    if (march_needed(S, S.inv + 12 * shape, q, ro, rd, best, o, d, start, end_c)) {
                        m.begin(q, o, d, start, end_c, S.march_G[k], S.march_F[k], false);
                        marching = true;
                        if (COUNT) c.march_rays++;
                        if (m.phase() == RT_PHASE_END) finish_shape();   // an empty range, or depth 0
                    }
                }
                // again, as long as the filter leaves lanes empty (the votes at the top decide)
                const unsigned still = __ballot_sync(FULL, !marching && !exhausted);
                if (still != 0 && __popc(still) >= RT_MARCH_REFILL_MIN) continue;
            }
        }
        if (__ballot_sync(FULL, marching) == 0) {
            if (__ballot_sync(FULL, have || !exhausted) == 0) break;
            continue;
        }
        // ---- marching: the warp votes between the expensive exact-jump attempt and the cheap literal
        //      steps, so that attempts run with many lanes at once ---------------------------------------
        int ph = marching ? m.phase() : -1;
        if (ph == RT_PHASE_END) {
            finish_shape();
            ph = -1;
        }
        const unsigned want_attempt = __ballot_sync(FULL, ph == RT_PHASE_ATTEMPT);
        const unsigned want_literal = __ballot_sync(FULL, ph == RT_PHASE_LITERAL);
        if (want_attempt && (want_literal == 0 || __popc(want_attempt) >= RT_MARCH_ATTEMPT_MIN)) {
            // (Letting the literal-phase lanes take steps inside the attempt's loops -- coop_advance's co_work
            // hook -- was measured: the longer loop bodies cost more than the idle lanes, 4.1 -> 4.65 ms.)
            typename Marcher<KIND, COUNT>::Plan pl;
            long long mj = 0;
            if (ph == RT_PHASE_ATTEMPT) mj = m.attempt_plan(pl);
            const unsigned jumping = __ballot_sync(FULL, mj > 0);
            if (jumping) {
                double nt = 0.0;
                D3 np = mk(0.0, 0.0, 0.0);
                coop_advance(jumping, mj, m.t, m.step, m.p, m.sd, nt, np, s_owner, []() {});
                if (mj > 0) m.attempt_land(pl, nt, np);
            }
        } else if (want_literal) {
            if (ph == RT_PHASE_LITERAL) {
#pragma unroll 1
                for (int rep = 0; rep < RT_MARCH_LITERAL_BURST; rep++) {
                    m.literal();
                    if (m.phase() != RT_PHASE_LITERAL) break;
                }
            }
        }
    }
    if (COUNT) flush_counters(c, g_counters);
}

int rt_march_occupancy() {
    int b = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_march<RT_SURF_HEART, false>, 128, 0);
    return std::max(b, 1);
}

template <int K_>
static void launch_kind(const MarchLaunch& ml) {
    if (ml.count)
        k_march<K_, true><<<ml.grid, 128, 0, ml.stream>>>(ml.ds, ml.kind_mask, ml.in, ml.hq, ml.march_count, ml.head, ml.counters, ml.tune);
    else
        k_march<K_, false><<<ml.grid, 128, 0, ml.stream>>>(ml.ds, ml.kind_mask, ml.in, ml.hq, ml.march_count, ml.head, ml.counters, ml.tune);
}

// K3a: the miss proof of rt_march.cuh (3) for every queued (ray, marched shape) pair, one entry per thread, before the
// marching kernels see the queue: straight-line code (ray -> object space, bounding chord, the surface polynomial along
// the ray, its Bernstein hull) that runs with full warps, where the same test inside the persistent marcher runs with
// whatever lanes happen to be starting a shape.  A proven miss clears the shape's bit in the entry's mask; the entries
// that keep a bit are written, compacted, to the filtered queue (hq.fq_slot / fq_mask, one atomic per warp), which is
// what the marching kernels then read.  (The proof is made for the chord clipped by the best hit known NOW; a later
// kind pass can only shorten that chord.)
template <int KIND, bool COUNT>
__device__ __forceinline__ bool filter_proves_miss(const double* q, D3 o, D3 d, double start, double end_c, double G, double F,
                                                   DevCounters& c) {
    Marcher<KIND, COUNT> m;
    m.begin(q, o, d, start, end_c, G, F);
    if (m.phase() != RT_PHASE_END || m.finish() != RT_MARCH_MISS) return false;
    if (COUNT) {
        c.march_rays++;
        c.march_steps += m.n;
        for (int k = 0; k < 8; k++) c.march_prof[k] += m.prof[k];
    }
    return true;
}
template <bool COUNT>
__global__ void __launch_bounds__(128)
k_march_filter(DevScene S, PathQueue in, HitQueue hq, const uint32_t* __restrict__ march_count, uint32_t* filtered_count,
               DevCounters* g_counters) {
    DevCounters c = {};
    const uint32_t n = *march_count;
    const uint32_t n_round = (n + 31u) & ~31u;   // whole warps stay converged for queue_append
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n_round; j += stride) {
        const bool valid = j < n;
        const uint32_t slot = valid ? hq.mq_slot[j] : 0u;
        const uint32_t mask0 = valid ? hq.mq_mask[j] : 0u;
        uint32_t mask = mask0, keep = 0;
        double best = 0.0;
        D3 ro = mk(0.0, 0.0, 0.0), rd = mk(0.0, 0.0, 0.0);
        if (valid) {
            best = hq.t[slot];
            ro = mk(in.ox[slot], in.oy[slot], in.oz[slot]);
            rd = mk(in.dx[slot], in.dy[slot], in.dz[slot]);
        }
        while (mask) {
            const int k = __ffs(mask) - 1;
            mask &= mask - 1;
            const int shape = S.march_index[k];
            const double* q = S.params + RT_SHAPE_PARAMS * shape;
            D3 o, d;
            double start, end_c;
            if (!march_needed(S, S.inv + 12 * shape, q, ro, rd, best, o, d, start, end_c)) continue;
            const double G = S.march_G[k], F = S.march_F[k];
            bool miss;
            switch ((int)q[0]) {
                case RT_SURF_HEART: miss = filter_proves_miss<RT_SURF_HEART, COUNT>(q, o, d, start, end_c, G, F, c); break;
                case RT_SURF_SINE: miss = filter_proves_miss<RT_SURF_SINE, COUNT>(q, o, d, start, end_c, G, F, c); break;
                case RT_SURF_STAR: miss = filter_proves_miss<RT_SURF_STAR, COUNT>(q, o, d, start, end_c, G, F, c); break;
                case RT_SURF_DUPIN: miss = filter_proves_miss<RT_SURF_DUPIN, COUNT>(q, o, d, start, end_c, G, F, c); break;
                case RT_SURF_HUNTS: miss = filter_proves_miss<RT_SURF_HUNTS, COUNT>(q, o, d, start, end_c, G, F, c); break;
                default: miss = filter_proves_miss<RT_SURF_CUSHION, COUNT>(q, o, d, start, end_c, G, F, c); break;
            }
            if (!miss) keep |= 1u << k;
        }
        // what is left goes to the compacted queue the marching kernels read (they would otherwise fetch and skip
        // the emptied entries -- more than half of them on cornell_box)
        const uint32_t at = queue_append(keep != 0, filtered_count);
        if (keep != 0) {
            hq.fq_slot[at] = slot;
            hq.fq_mask[at] = keep;
        }
    }
    if (COUNT) flush_counters(c, g_counters);
}

void rt_launch_march_filter(const MarchLaunch& ml) {
    if (ml.count) k_march_filter<true><<<ml.grid_filter, 128, 0, ml.stream>>>(ml.ds, ml.in, ml.hq, ml.march_count, ml.filtered_count, ml.counters);
    else k_march_filter<false><<<ml.grid_filter, 128, 0, ml.stream>>>(ml.ds, ml.in, ml.hq, ml.march_count, ml.filtered_count, ml.counters);
}

void rt_launch_march(const MarchLaunch& ml) {
    switch (ml.kind) {
        case RT_SURF_HEART: launch_kind<RT_SURF_HEART>(ml); break;
        case RT_SURF_SINE: launch_kind<RT_SURF_SINE>(ml); break;
        case RT_SURF_STAR: launch_kind<RT_SURF_STAR>(ml); break;
        case RT_SURF_DUPIN: launch_kind<RT_SURF_DUPIN>(ml); break;
        case RT_SURF_HUNTS: launch_kind<RT_SURF_HUNTS>(ml); break;
        default: launch_kind<RT_SURF_CUSHION>(ml); break;
    }
}
