// Device-resident scene (structure of arrays), winner finalisation, textures, materials and the
// one-step integrator shared by every kernel of the core.  FP64, no FMA contraction (see rt_math.cuh).
#pragma once
#include "rt_math.cuh"
#include "rt_march.cuh"
#include "rt_cull.cuh"

namespace rt {

struct DevImage {
    uint32_t width, height;
    const uint8_t* rgba;
};

// Flat scene in HBM.  inv/dir: [n][12] rows 0..2 of InversableTransform.inverse/.direct;
// params: [n][8]; everything is read-only for the lifetime of the rt_scene.
struct DevScene {
    int n_shapes;
    const double* inv;
    const double* dir;
    const double* params;
    const uint8_t* kind;
    const uint8_t* flags;
    const uint32_t* material;
    const rt_material* materials;
    const uint8_t* mat_bin;     // [n_materials] shade key of a material: its (kind, root texture kind) bin (k_shade)
    const rt_texture* textures;
    const DevImage* images;
    const rt_perlin* noise;
    // indices of the RT_SHAPE_MARCH shapes (they are few; kernels that split marching out of the
    // analytic loop walk this list)
    int n_march;
    const int* march_index;
    const double* march_G;      // [n_march] bound of |grad f| over the marching region (inf: never skip)
    const double* march_F;      // [n_march] bound of sum |monomials of f| over the region (rounding of f)
    const float4* march_cull;   // [n_march] conservative ball around the marching bound (rt_cull.cuh)
    // conservative cull tree (rt_cull.cuh, CullTree): ctab = [roots][groups][16 leaves per group][flat list],
    // cids = shape index of every leaf / flat slot (-1 = padding)
    int n_roots, n_groups, n_flat, n_flat_real;
    const float4* ctab;
    // levels above the roots (CullTree::upper): level l at cupper[upper_off[l]], l = 1 .. n_upper
    int n_upper, upper_off[RT_CULL_UPPER_MAX + 1];
    const float4* cupper;
    const int* cids;
    // per shape (RT_ISECT_VERIFY): its own leaf entry and its group (-1 flat list, -2 not analytic)
    const float4* cull;
    const int* cull_group;
    __host__ __device__ int ctab_entries() const { return n_roots + n_groups + RT_CULL_GROUP * n_groups + n_flat; }
    // FlatRec: one record of RT_FLAT_REC doubles per flat-list entry, in flat-list order -- [0..11] inverse rows,
    // [12..15] params 0..3 (Rectangle bounds), [16] = {int shape index, int kind}, [17] padding (144 B, 16-byte
    // aligned).  n_frec = n_flat_real, or 0 when the flat list is too long to be worth staging.
    int n_frec;
    const double* frec;
};
#define RT_FLAT_REC 18
#define RT_FLAT_REC_MAX 64

// optional work counters (rt_stats); enabled per launch by a template flag
struct DevCounters {
    unsigned long long segments, shape_tests, cull_tests, march_steps, march_rays;
    unsigned long long march_long_rays;  // marched rays that needed more than 2048 evaluations
    unsigned long long march_max_evals;  // most evaluations any single marched ray needed
    unsigned long long verify_rays;         // RT_ISECT_VERIFY: rays whose FAST result differs from BRUTE
    unsigned long long verify_false_culls;  // RT_ISECT_VERIFY: (ray, shape) pairs culled although the exact test hits
    unsigned long long march_prof[8];       // k_march: literal steps at level 0 / deeper, exact jumps, bound hops, misses by hull / by hops
};

struct HitRec {  // RayHit, src/world/ray.rs:21-29
    D3 point, normal;
    double t, u, v;
    bool front;
    int shape;
};

// Rebuild the winner's RayHit from (shape, t, ray): Shape::ray_hit_transformed
// (src/world/shapes/mod.rs:112-124) around the tail of each ray_intersect and RayHit::new /
// set_normal (src/world/ray.rs:32-64).
// want_uv = false: the caller knows (u, v) will not be read (material_reads_uv) -- the Sphere's acos / atan2 and the
// Rectangle's two divisions are skipped and u = v = 0.
__device__ inline void finalize_hit(const DevScene& S, int i, double t, D3 ro, D3 rd, HitRec& h, bool want_uv = true) {
    const double* inv = S.inv + 12 * i;
    const double* q = S.params + RT_SHAPE_PARAMS * i;
    const double PI = 3.14159265358979323846264338327950288;
    D3 o = xf_point(inv, ro);   // inverse_transform_ray, src/algebra/transform.rs:32-37
    D3 d = xf_vector(inv, rd);
    D3 p = o + d * t;
    D3 n;
    double u = 0.0, v = 0.0;
    switch (S.kind[i]) {
        case RT_SHAPE_SPHERE: {  // shapes/mod.rs:358-373
            n = (S.flags[i] & RT_SHAPE_FLAG_INVERSE_NORMAL) ? -p : p;
            if (want_uv) {
                double theta = acos(-p.y);
                double phi = atan2(-p.z, p.x) + PI;
                u = phi / (2.0 * PI);
                v = theta / PI;
            }
            break;
        }
        case RT_SHAPE_CUBE: {  // :263-283
            double ax = fabs(p.x), ay = fabs(p.y), az = fabs(p.z);
            double max_c = max3(ax, ay, az);
            if (max_c == ax) { n = mk(p.x, 0.0, 0.0); u = p.y; v = p.z; }
            else if (max_c == ay) { n = mk(0.0, p.y, 0.0); u = p.x; v = p.z; }
            else { n = mk(0.0, 0.0, p.z); u = p.x; v = p.y; }
            break;
        }
        case RT_SHAPE_RECTANGLE: {  // :191-201
            n = mk(0.0, 0.0, 1.0);
            if (want_uv) {
                u = (p.x - q[0]) / (q[2] - q[0]);
                v = (p.y - q[1]) / (q[3] - q[1]);
            }
            break;
        }
        case RT_SHAPE_TORUS: {  // shapes/mod.rs:453-468
            n = p - normalize(mk(p.x, p.y, 0.0)) * q[0];
            if (want_uv) {
                const double theta = asin(p.z / q[1]);
                const double phi = acos(p.z / (q[0] + q[1] * cos(theta))) + PI;
                u = phi / (2.0 * PI);
                v = theta / PI;
            }
            break;
        }
        default: {  // RT_SHAPE_MARCH, ray_marching.rs:59-61
            n = surface_gradient(q, p);
            int sk = (int)q[0];
            if (sk == RT_SURF_DUPIN || sk == RT_SURF_HUNTS || sk == RT_SURF_CUSHION) { u = p.x; v = p.y; }
            break;
        }
    }
    D3 n_obj = normalize(n);                           // RayHit::new, ray.rs:42-45
    h.point = xf_point(S.dir + 12 * i, p);             // shapes/mod.rs:117
    D3 n_w = xf_normal(inv, n_obj);                    // shapes/mod.rs:118
    bool front = dot(n_w, rd) < 0.0;                   // set_normal, ray.rs:60-64
    h.normal = normalize(front ? n_w : -n_w);
    h.front = front;
    h.t = t;
    h.u = u;
    h.v = v;
    h.shape = i;
}

// One candidate test: Shape::ray_hit for shape i with the current max_t (shapes/mod.rs:126-137).
// `m` points at the shape's inverse rows (shared or global memory).
template <bool COUNT>
__device__ __forceinline__ bool shape_candidate(const DevScene& S, int i, int kind, const double* m, D3 ro, D3 rd,
                                                double min_t, double max_t, double& t, DevCounters& c) {
    D3 o = xf_point(m, ro);
    D3 d = xf_vector(m, rd);
    if (COUNT) c.shape_tests++;
    if (kind == RT_SHAPE_SPHERE) return sphere_candidate(o, d, min_t, max_t, t);
    if (kind == RT_SHAPE_CUBE) return cube_candidate(o, d, min_t, max_t, t);
    if (kind == RT_SHAPE_RECTANGLE) return rect_candidate(S.params + RT_SHAPE_PARAMS * i, o, d, min_t, max_t, t);
    if (kind == RT_SHAPE_TORUS) return torus_candidate(S.params + RT_SHAPE_PARAMS * i, o, d, min_t, max_t, t);
    unsigned long long ev = 0;
    bool ok = march_candidate(S.params + RT_SHAPE_PARAMS * i, o, d, min_t, max_t, t, ev);
    if (COUNT) {
        c.march_steps += ev;
        c.march_rays += 1;  // counts bound hits + misses alike; refined by the split kernels
    }
    return ok;
}

// ShapeCollection::ray_intersect (src/world/shapes/mod.rs:573-597): index order, shrinking max_t.
// s_inv / s_kind: the shape list staged in shared memory (or the global arrays when it does not fit).
template <bool COUNT>
__device__ __forceinline__ void nearest_hit_brute(const DevScene& S, D3 ro, D3 rd, double min_t, double max_t,
                                                  double& best_t, int& best_i, DevCounters& c) {
    double min_distance = max_t;
    int winner = -1;
    const int n = S.n_shapes;
    for (int i = 0; i < n; i++) {
        double t;
        if (shape_candidate<COUNT>(S, i, S.kind[i], S.inv + 12 * i, ro, rd, min_t, min_distance, t, c)) {
            min_distance = t;
            winner = i;
        }
    }
    if (COUNT) c.segments++;
    best_t = min_distance;
    best_i = winner;
}

// The same nearest hit, reorganised (RT_ISECT_FAST and the wavefront renderer):
//   1. the analytic shapes in index order with the shrinking max_t (identical arithmetic);
//   2. the ray-marched shapes afterwards, skipped when their bounding chord starts behind the best
//      hit so far, clipped two steps past it otherwise, and marched with exact skipping (rt_march.cuh).
// Every candidate t is independent of max_t except for acceptance (SURVEY A.3), so the sequential
// loop's result is the lexicographic minimum of (t, -index); step 2 applies that rule explicitly.
// The two inputs on which the sequential loop is NOT a pure arg-min — a Sphere hit through the
// unchecked D == 0 branch and a NaN t — are detected ("degenerate") and replayed through
// nearest_hit_brute.

// the shape list as the analytic loop sees it: the cull table, staged in dynamic shared memory when it
// fits (rt_core.cu: stage_scene), else read from global memory.  The shared copy is addressed through
// the extern array itself so that the compiler emits LDS rather than generic loads.
extern __shared__ __align__(16) unsigned char rt_smem_raw[];
struct Staged {
    bool smem;
};

// one exact candidate test of analytic shape i (kind != MARCH) against the current best.  mp: the shape's
// inverse rows, q: its params; NC = read them through the non-coherent path (global arrays) or with plain
// loads (records staged in shared memory)
template <bool NC>
__device__ __forceinline__ double2 ld2(const double2* p) {
    if (NC) return __ldg(p);
    return *p;
}
template <bool COUNT, bool NC>
__device__ __forceinline__ void analytic_test_at(int i, int kind, const double2* mp, const double* q, D3 ro, D3 rd,
                                                 double min_t, double& best, int& winner, bool& degenerate,
                                                 DevCounters& c) {
    if (COUNT) c.shape_tests++;
    double t;
    bool ok;
    if (kind == RT_SHAPE_TORUS) {
        // Torus (shapes/mod.rs:429-476): the complex quartic solver stays out of this loop (its call frame cost
        // every scene 240 B of spills in k_extend).  A ray whose line touches the torus's bounding ball is replayed
        // through the literal loop instead (k_replay -> nearest_hit_brute -> torus_candidate), like a degenerate one.
        degenerate = true;
        return;
    }
    if (kind == RT_SHAPE_RECTANGLE) {
        // Rectangle::ray_intersect (shapes/mod.rs:181-190) needs only o.z, d.z to reject most rays: row 2 of the
        // inverse first, the other rows when x = -o.z / d.z is in range (same operations, same order as
        // xf_point / xf_vector + rect_candidate, so the same bits).
        const double2 r20 = ld2<NC>(mp + 4), r21 = ld2<NC>(mp + 5);
        const double oz = ro.x * r20.x + ro.y * r20.y + ro.z * r21.x + r21.y;
        const double dz = rd.x * r20.x + rd.y * r20.y + rd.z * r21.x;
        // o.z and d.z finite, non-zero and of the same sign: x = -o.z / d.z is negative (or -0), below min_t > 0
        const double sgn = oz * dz;
        if (min_t > 0.0 && sgn > 0.0 && sgn < INFINITY) return;
        const double x = -oz / dz;
        if (x < min_t || x > best) return;
        const double2 r00 = ld2<NC>(mp), r01 = ld2<NC>(mp + 1), r10 = ld2<NC>(mp + 2), r11 = ld2<NC>(mp + 3);
        const double ox = ro.x * r00.x + ro.y * r00.y + ro.z * r01.x + r01.y;
        const double oy = ro.x * r10.x + ro.y * r10.y + ro.z * r11.x + r11.y;
        const double dx = rd.x * r00.x + rd.y * r00.y + rd.z * r01.x;
        const double dy = rd.x * r10.x + rd.y * r10.y + rd.z * r11.x;
        const double px = ox + dx * x, py = oy + dy * x;
        if (px < q[0] || px > q[2] || py < q[1] || py > q[3]) return;
        t = x;
        ok = true;
    } else {
        double m[12];
#pragma unroll
        for (int k = 0; k < 6; k++) {
            double2 v = ld2<NC>(mp + k);
            m[2 * k] = v.x;
            m[2 * k + 1] = v.y;
        }
        D3 o = xf_point(m, ro);
        D3 d = xf_vector(m, rd);
        if (kind == RT_SHAPE_SPHERE) ok = sphere_candidate(o, d, min_t, best, t, &degenerate);
        else ok = cube_candidate(o, d, min_t, best, t);
    }
    if (ok) {  // ok means t <= best (or a degenerate candidate); shapes are not visited in index order, so the
               // loop's "later shape wins ties" is explicit
        if (t != t) degenerate = true;
        if (t < best || i > winner || degenerate) {
            best = t;
            winner = i;
        }
    }
}
template <bool COUNT>
__device__ __forceinline__ void analytic_test(const DevScene& S, int i, D3 ro, D3 rd, double min_t, double& best,
                                              int& winner, bool& degenerate, DevCounters& c) {
    analytic_test_at<COUNT, true>(i, S.kind[i], reinterpret_cast<const double2*>(S.inv + 12 * i),  // rows are 96 B
                                  S.params + RT_SHAPE_PARAMS * i, ro, rd, min_t, best, winner, degenerate, c);
}

// step 1.  Returns true when the ray is degenerate.  FP32 culling first (rt_cull.cuh): the flat list,
// then roots -> groups -> leaves of the tree; each lane runs the exact test on its own survivors.
// ANY (any_hit_fast): return at the first exact test that accepts the ray, winner >= 0.  Until then best == max_t, so
// every test runs at the caller's bound.
template <bool COUNT, bool SMEM, bool ANY = false>
__device__ __forceinline__ bool analytic_nearest_impl(const DevScene& S, const CullRay& cr, D3 ro, D3 rd, double min_t,
                                                      double max_t, double& best, int& winner, DevCounters& c) {
    best = max_t;
    winner = -1;
    bool degenerate = false;
    const float4* roots = SMEM ? reinterpret_cast<const float4*>(rt_smem_raw) : S.ctab;
    const float4* groups = roots + S.n_roots;
    const float4* leaves = groups + S.n_groups;
    const float4* flat = leaves + RT_CULL_GROUP * S.n_groups;
    const int* flat_ids = S.cids + RT_CULL_GROUP * S.n_groups;
    if (S.n_frec > 0) {
        // the flat list through its records: entry j's exact test reads frec[j] (staged behind the table), and
        // an entry that is never culled (w = +inf: Rectangles, ill-conditioned transforms) skips the pre-test,
        // whose answer is known -- the same decisions as the loop below
        const double* frec = SMEM ? reinterpret_cast<const double*>(rt_smem_raw + sizeof(float4) * S.ctab_entries())
                                  : S.frec;
        for (int j = 0; j < S.n_frec; j++) {
            const float4 e = flat[j];
            if (e.w != INFINITY && !cull_pass(cr, e)) continue;
            const double* r = frec + RT_FLAT_REC * j;
            const int2 tag = *reinterpret_cast<const int2*>(r + 16);
            if (SMEM) analytic_test_at<COUNT, false>(tag.x, tag.y, reinterpret_cast<const double2*>(r), r + 12, ro, rd, min_t, best, winner, degenerate, c);
            else analytic_test_at<COUNT, true>(tag.x, tag.y, reinterpret_cast<const double2*>(r), r + 12, ro, rd, min_t, best, winner, degenerate, c);
            if (ANY && winner >= 0) {
                if (COUNT) c.cull_tests += j + 1;
                return degenerate;
            }
        }
    } else
    for (int f0 = 0; f0 < S.n_flat; f0 += 32) {
        const int nf = min(32, S.n_flat - f0);  // a multiple of 8
        uint32_t mask = 0;
#pragma unroll 8
        for (int j = 0; j < nf; j++)
            if (cull_pass(cr, flat[f0 + j])) mask |= 1u << j;
        while (mask) {
            const int j = __ffs(mask) - 1;
            mask &= mask - 1;
            // (a NaN ray passes every pre-test, the padding entries' too: their id is -1)
            const int id = __ldg(flat_ids + f0 + j);
            if (id >= 0) analytic_test<COUNT>(S, id, ro, rd, min_t, best, winner, degenerate, c);
            if (ANY && winner >= 0) {
                if (COUNT) c.cull_tests += min(f0 + nf, S.n_flat_real);
                return degenerate;
            }
        }
    }
    if (COUNT) c.cull_tests += S.n_flat_real;
    for (int r = 0; r < S.n_roots; r++) {
        if (S.n_upper > 0) {
            // arbitrary depth: entering the range of an upper node (32^l roots, aligned), test it -- top level first --
            // and skip the whole range when the line misses its ball
            bool skipped = false;
            for (int l = S.n_upper; l >= 1 && !skipped; l--) {
                const int span = 1 << (5 * l);
                if ((r & (span - 1)) != 0) continue;
                if (COUNT) c.cull_tests++;
                if (!cull_pass_node(cr, __ldg(S.cupper + S.upper_off[l] + (r >> (5 * l))))) {
                    r += span - 1;   // (the loop's r++ completes the skip)
                    skipped = true;
                }
            }
            if (skipped) continue;
        }
        if (COUNT) c.cull_tests++;
        if (!cull_pass_node(cr, roots[r])) continue;
        const int g0 = RT_CULL_ROOT_FANOUT * r;
        const int ng = min(RT_CULL_ROOT_FANOUT, S.n_groups - g0);  // a multiple of 8
        uint32_t gmask = 0;
#pragma unroll 8
        for (int j = 0; j < ng; j++)
            if (cull_pass_node(cr, groups[g0 + j])) gmask |= 1u << j;
        if (COUNT) c.cull_tests += ng + RT_CULL_GROUP * __popc(gmask);
        while (gmask) {
            const int g = g0 + __ffs(gmask) - 1;
            gmask &= gmask - 1;
            const float4* lv = leaves + RT_CULL_GROUP * g;
            uint32_t mask = 0;
#pragma unroll
            for (int j = 0; j < RT_CULL_GROUP; j++)
                if (cull_pass(cr, lv[j])) mask |= 1u << j;
            while (mask) {
                const int j = __ffs(mask) - 1;
                mask &= mask - 1;
                const int id = __ldg(S.cids + RT_CULL_GROUP * g + j);
                if (id >= 0) analytic_test<COUNT>(S, id, ro, rd, min_t, best, winner, degenerate, c);
                if (ANY && winner >= 0) return degenerate;
            }
        }
    }
    return degenerate;
}
template <bool COUNT, bool ANY = false>
__device__ __forceinline__ bool analytic_nearest(const DevScene& S, const Staged& st, const CullRay& cr, D3 ro, D3 rd,
                                                 double min_t, double max_t, double& best, int& winner, DevCounters& c) {
    if (st.smem) return analytic_nearest_impl<COUNT, true, ANY>(S, cr, ro, rd, min_t, max_t, best, winner, c);
    return analytic_nearest_impl<COUNT, false, ANY>(S, cr, ro, rd, min_t, max_t, best, winner, c);
}

// does marched shape number k (position in S.march_index) have to be marched for this ray, given the
// best hit so far?  On true, o/d are the object-space ray and [start, end_c] the (clipped) chord.
__device__ __forceinline__ bool march_needed(const DevScene& S, const double* m, const double* q, D3 ro, D3 rd,
                                             double best, D3& o, D3& d, double& start, double& end_c) {
    o = xf_point(m, ro);
    d = xf_vector(m, rd);
    double end;
    if (!march_bound(q, o, d, start, end)) return false;
    const double step = q[1];
    end_c = end;
    if (step > 0.0) {
        // every candidate lies at or beyond start: a chord that starts past the best hit cannot win; one that starts
        // exactly AT it still can (t == best, later shape index wins the tie); a NaN start is dropped as before
        if (!(start <= best)) return false;
        end_c = fmin(end, best + 2.0 * step);        // a hit found later than this cannot win
    }
    return true;
}

// step 2 for one marched shape.  Returns true when the ray turned out degenerate.
template <bool COUNT>
__device__ __forceinline__ bool march_shape_update(const DevScene& S, const CullRay& cr, const double* s_inv, int k,
                                                   D3 ro, D3 rd, double min_t, double max_t, double& best, int& winner,
                                                   DevCounters& c) {
    if (COUNT) c.cull_tests++;
    if (!cull_pass(cr, S.march_cull[k])) return false;  // the line misses the marching bound: None
    const int i = S.march_index[k];
    const double* q = S.params + RT_SHAPE_PARAMS * i;
    D3 o, d;
    double start, end_c;
    if (COUNT) c.shape_tests++;
    if (!march_needed(S, s_inv + 12 * i, q, ro, rd, best, o, d, start, end_c)) return false;
    if (COUNT) c.march_rays++;
    unsigned long long ev = 0;
    double t;
    bool ok = march_candidate_skip(q, o, d, start, end_c, min_t, max_t, S.march_G[k], S.march_F[k], t, ev);
    if (COUNT) {
        c.march_steps += ev;
        if (ev > 2048) c.march_long_rays++;
        if (ev > c.march_max_evals) c.march_max_evals = ev;
    }
    if (ok) {
        if (t != t) return true;
        if (t < best || (t == best && i > winner)) {
            best = t;
            winner = i;
        }
    }
    return false;
}

template <bool COUNT>
__device__ __forceinline__ void nearest_hit_fast(const DevScene& S, const Staged& st, D3 ro, D3 rd, double min_t,
                                                 double max_t, double& best_t, int& best_i, DevCounters& c) {
    double best;
    int winner;
    const CullRay cr = make_cull_ray(ro.x, ro.y, ro.z, rd.x, rd.y, rd.z);
    bool degenerate = analytic_nearest<COUNT>(S, st, cr, ro, rd, min_t, max_t, best, winner, c);
    for (int k = 0; k < S.n_march && !degenerate; k++)
        degenerate = march_shape_update<COUNT>(S, cr, S.inv, k, ro, rd, min_t, max_t, best, winner, c);
    if (degenerate) {
        nearest_hit_brute<COUNT>(S, ro, rd, min_t, max_t, best_t, best_i, c);
        return;
    }
    if (COUNT) c.segments++;
    best_t = best;
    best_i = winner;
}

// Any-hit (rt_occluded_batch): does some shape accept the ray at (min_t, max_t)?  The literal loop's max_t only
// shrinks at an acceptance, so its first acceptance is tested at max_t, and it returns a hit iff some shape accepts at
// max_t -- a Sphere D == 0 hit and a NaN t included.  So the answer is nearest_hit_brute's `index != -1`, in any
// order of the shapes, and the walk stops at the first acceptance.
template <bool COUNT>
__device__ __forceinline__ bool any_hit_brute(const DevScene& S, D3 ro, D3 rd, double min_t, double max_t,
                                              DevCounters& c) {
    for (int i = 0; i < S.n_shapes; i++) {
        double t;
        if (shape_candidate<COUNT>(S, i, S.kind[i], S.inv + 12 * i, ro, rd, min_t, max_t, t, c)) return true;
    }
    return false;
}

// The same answer through the cull tree: the analytic shapes first, then the marched ones (exact skipping, chords
// that start past max_t skipped), each stopping at the first acceptance.  A degenerate ray (a Sphere D == 0 branch or
// a NaN t the analytic pass did not accept, a Torus ball touched, a NaN marched t) finishes through the literal loop.
// A NaN bound does too: march_needed drops every chord against it, the literal loop does not.  The marcher runs without
// the Bernstein miss proof, like k_intersect_batch's: on a B200 the proof made dupin's shadow rays 10 % slower (424.6 ->
// 383.9 Mrays/s) and the bench trio's config 2 rays 7 % faster (2381 -> 2540), so the simpler form stays.
template <bool COUNT>
__device__ __forceinline__ bool any_hit_fast(const DevScene& S, const Staged& st, D3 ro, D3 rd, double min_t,
                                             double max_t, DevCounters& c) {
    if (max_t != max_t || min_t != min_t) return any_hit_brute<COUNT>(S, ro, rd, min_t, max_t, c);
    double best;
    int winner;
    const CullRay cr = make_cull_ray(ro.x, ro.y, ro.z, rd.x, rd.y, rd.z);
    bool degenerate = analytic_nearest<COUNT, true>(S, st, cr, ro, rd, min_t, max_t, best, winner, c);
    if (winner >= 0) return true;
    for (int k = 0; k < S.n_march && !degenerate; k++) {
        degenerate = march_shape_update<COUNT>(S, cr, S.inv, k, ro, rd, min_t, max_t, best, winner, c);
        if (winner >= 0) return true;
    }
    if (degenerate) return any_hit_brute<COUNT>(S, ro, rd, min_t, max_t, c);
    return false;
}

// ------------------------------------------------------------------------------------------------
// textures — src/world/texture.rs:17-116
// ------------------------------------------------------------------------------------------------
// Perlin::noise, src/algebra/noise.rs:43-73: gradient noise over the unit cell of p, corners in
// multi_cartesian_product order (last index fastest), terms summed in that order from 0.0
__device__ inline double perlin_noise(const rt_perlin& pn, D3 p) {
    const double fx = floor(p.x), fy = floor(p.y), fz = floor(p.z);
    auto as_i32 = [](double v) -> int {  // `as i32`: saturating, NaN -> 0
        if (v != v) return 0;
        if (v <= -2147483648.0) return (int)0x80000000;
        if (v >= 2147483647.0) return 2147483647;
        return (int)v;
    };
    const unsigned x = (unsigned)as_i32(fx), y = (unsigned)as_i32(fy), z = (unsigned)as_i32(fz);
    const double u = p.x - fx, v = p.y - fy, w = p.z - fz;
    const double u2 = u * u * (3.0 - 2.0 * u);
    const double v2 = v * v * (3.0 - 2.0 * v);
    const double w2 = w * w * (3.0 - 2.0 * w);
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const int d0 = (k >> 2) & 1, d1 = (k >> 1) & 1, d2 = k & 1;
        const rt_vec3 c = pn.ranvec[pn.perm_x[(d0 + x) & 255u] ^ pn.perm_y[(d1 + y) & 255u] ^ pn.perm_z[(d2 + z) & 255u]];
        const double fi = (double)d0, fj = (double)d1, fk = (double)d2;
        const double dotp = c.x * (u - fi) + c.y * (v - fj) + c.z * (w - fk);
        sum = sum + (fi * u2 + (double)(1 - d0) * (1.0 - u2)) * (fj * v2 + (double)(1 - d1) * (1.0 - v2)) *
                        (fk * w2 + (double)(1 - d2) * (1.0 - w2)) * dotp;
    }
    return sum;
}
// Perlin::turb, :75-86.  The reference's scan evaluates noise(&p) -- the ORIGINAL point, not the doubled
// temp_p -- at every octave, so the result is |sum_i 2^-i noise(p)| with the sum's own roundings.
__device__ inline double perlin_turb(const rt_perlin& pn, D3 p, int depth) {
    const double n = perlin_noise(pn, p);
    double sum = 0.0, weight = 1.0;
    for (int i = 0; i < depth; i++) {
        sum = sum + weight * n;
        weight *= 0.5;
    }
    return fabs(sum);
}

__device__ inline D3 texture_value(const DevScene& S, uint32_t tex, double u, double v, D3 p) {
    const double PI = 3.14159265358979323846264338327950288;
    for (int depth = 0; depth <= RT_TEX_MAX_DEPTH; depth++) {
        const rt_texture& t = S.textures[tex];
        if (t.kind == RT_TEX_SOLID) return mk(t.color.x, t.color.y, t.color.z);
        if (t.kind == RT_TEX_CHECKER) {  // :40-51
            double sines = sin(t.color.x * p.x) * sin(t.color.y * p.y) * sin(t.color.z * p.z);
            tex = sines < 0.0 ? t.odd : t.even;
        } else if (t.kind == RT_TEX_UV_CHECKER) {  // :78-88 (v pairs with multipliers.0)
            double sines = sin(v * t.color.x * PI) * sin(u * t.color.y * PI);
            tex = sines < 0.0 ? t.odd : t.even;
        } else if (t.kind == RT_TEX_IMAGE) {  // :98-117
            const DevImage& im = S.images[t.image];
            double uu = isnan(u) ? u : fmin(fmax(u, 0.0), 1.0);
            double vc = isnan(v) ? v : fmin(fmax(v, 0.0), 1.0);
            double vv = 1.0 - vc;
            double fx = uu * (double)im.width, fy = vv * (double)im.height;
            // `as u32`: saturating, NaN -> 0.  get_pixel panics at x == width; clamp instead (SURVEY A.10)
            uint32_t x = isnan(fx) ? 0u : (fx <= 0.0 ? 0u : (fx >= 4294967295.0 ? 4294967295u : (uint32_t)fx));
            uint32_t y = isnan(fy) ? 0u : (fy <= 0.0 ? 0u : (fy >= 4294967295.0 ? 4294967295u : (uint32_t)fy));
            if (x >= im.width) x = im.width - 1;
            if (y >= im.height) y = im.height - 1;
            const uint8_t* px = im.rgba + ((size_t)y * im.width + x) * 4;
            double color_scale = 1.0 / 255.0;
            return mk((double)px[0] * color_scale, (double)px[1] * color_scale, (double)px[2] * color_scale);
        } else if (t.kind == RT_TEX_NOISE) {  // NoiseTexture::value, :61-67
            const double k = 0.5 * (1.0 + sin(t.color.x * p.z + 10.0 * perlin_turb(S.noise[t.image], p, 7)));
            return mk(k * 1.0, k * 1.0, k * 1.0);
        } else {
            return mk(0.0, 0.0, 0.0);
        }
    }
    return mk(0.0, 0.0, 0.0);
}

// Dielectric::reflectance, src/world/material.rs:84-88; powi(5) = x * ((x*x)*(x*x))
__device__ __forceinline__ double reflectance(double cosine, double ref_index) {
    double r0 = (1.0 - ref_index) / (1.0 + ref_index);
    r0 = r0 * r0;
    double x = 1.0 - cosine;
    double x2 = x * x;
    double x5 = x * (x2 * x2);
    return r0 + (1.0 - r0) * x5;
}

// Material::scatter (src/world/material.rs:42-115).  Returns false when the material does not
// scatter (DiffuseLight, EmptyMaterial); then `atten` holds Material::emitted (:123-127).
// `ball`: random_in_unit_sphere drawn beforehand at the start of the event's stream (k_shade samples it
// warp-cooperatively, material_needs_ball says for which lanes), or nullptr to draw it here.
// Only texture lookups read the hit's (u, v), and a SolidColor root never does (texture.rs:17-24); Dielectric
// and EmptyMaterial have no texture at all.
__device__ __forceinline__ bool material_reads_uv(const DevScene& S, const rt_material& m) {
    if (m.kind == RT_MAT_DIELECTRIC || m.kind == RT_MAT_EMPTY) return false;
    return S.textures[m.texture].kind != RT_TEX_SOLID;
}
__device__ __forceinline__ bool material_needs_ball(const rt_material& m) {
    return m.kind == RT_MAT_LAMBERTIAN || (m.kind == RT_MAT_METAL && m.scalar != 0.0);
}
__device__ inline bool scatter_or_emit(const DevScene& S, const HitRec& h, D3 rd, PathRng& rng, D3& new_dir,
                                       D3& atten, const D3* ball = nullptr) {
    const rt_material m = S.materials[S.material[h.shape]];
    switch (m.kind) {
        case RT_MAT_LAMBERTIAN: {  // :42-53
            D3 direction = h.normal + (ball ? normalize(*ball) : random_unit(rng));
            if (approx_zero(direction.x) && approx_zero(direction.y) && approx_zero(direction.z)) direction = h.normal;
            new_dir = normalize(direction);  // Ray::new, ray.rs:12-17
            atten = texture_value(S, m.texture, h.u, h.v, h.point);
            return true;
        }
        case RT_MAT_METAL: {  // :64-75
            D3 reflected = reflect(rd, h.normal);
            D3 direction = (m.scalar == 0.0) ? reflected
                                             : reflected + m.scalar * (ball ? *ball : random_in_unit_sphere(rng));
            new_dir = normalize(direction);
            atten = texture_value(S, m.texture, h.u, h.v, h.point);
            return true;
        }
        case RT_MAT_DIELECTRIC: {  // :93-115
            double refract_ratio = h.front ? 1.0 / m.scalar : m.scalar;
            double cos_theta = dot(-rd, h.normal);
            double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
            D3 direction;
            if (refract_ratio * sin_theta > 1.0 || reflectance(cos_theta, refract_ratio) > rng.next())
                direction = reflect(rd, h.normal);
            else
                direction = refract(rd, h.normal, refract_ratio);
            new_dir = normalize(direction);
            atten = mk(1.0, 1.0, 1.0);
            return true;
        }
        case RT_MAT_DIFFUSE_LIGHT:
            atten = texture_value(S, m.texture, h.u, h.v, h.point);
            return false;
        default:
            atten = mk(0.0, 0.0, 0.0);
            return false;
    }
}

// The `atten` scatter_or_emit gives for the hit, without its random draws (the colour depends on the hit only):
// features frames record it.  A separate switch, so that scatter_or_emit's callers keep their generated code.
__device__ __forceinline__ D3 material_color(const DevScene& S, const HitRec& h) {
    const rt_material m = S.materials[S.material[h.shape]];
    switch (m.kind) {
        case RT_MAT_LAMBERTIAN:
        case RT_MAT_METAL:
        case RT_MAT_DIFFUSE_LIGHT:
            return texture_value(S, m.texture, h.u, h.v, h.point);
        case RT_MAT_DIELECTRIC:
            return mk(1.0, 1.0, 1.0);
        default:
            return mk(0.0, 0.0, 0.0);
    }
}

// Scene::background, src/world/mod.rs:199-202
__device__ __forceinline__ D3 sky(D3 rd) {
    double t = 0.5 * (rd.y + 1.0);
    return (1.0 - t) * mk(1.0, 1.0, 1.0) + t * mk(0.5, 0.7, 1.0);
}

}  // namespace rt
