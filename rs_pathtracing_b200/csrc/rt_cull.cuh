// Conservative FP32 bounding-ball cull in front of the exact FP64 shape tests.
//
// ShapeCollection::ray_intersect (src/world/shapes/mod.rs:573-597) tests every shape for every ray in
// FP64 (33 flop ray -> object space + 19 flop unit-sphere discriminant, Sphere::ray_intersect :330-356).
// A shape may be skipped for a ray iff the reference's test would return None for EVERY max_t; then
// skipping it leaves the sequential loop's state untouched and the result is bit-identical.
//
// Host side (cull_entry): for a Sphere / Cube with inverse rows [M | tv] the object-space ball |p'| <= ext
// (ext = 1 / sqrt 3) is, in world space, inside the ball  centre C = -M^-1 tv,  radius R = ext * ||M^-1||_2
// (Gershgorin bound of the spectral norm; exact for translate*rotate*scale).  It is derived from the
// INVERSE rows because those are what the exact test multiplies the ray with.
//
// Device side (cull_pass), FP32 with explicit FMAs, direction renormalised in FP32:
//     oc = C - o,  b = oc.d,  p = oc - b d,
//     reject  iff  |p|^2 > rhs,      rhs = 1.1 R^2 + 3B(|C|^2 + |o|^2)
// i.e. the test is on the LINE, not the half-line: a sphere behind the origin must not be culled, because
// the reference's D == 0 branch (src/world/shapes/mod.rs:343-344) accepts a tangent line without any
// range check, wherever the tangent point lies (tests: test_cull_is_conservative_on_fixture_scenes).
// Why this is conservative (u = 2^-24):
//   * every FP32 quantity above carries an absolute error <= 16u(|C| + |o| + |oc|) (input rounding, the
//     5u error of the renormalised direction, 3 FMA roundings), so a line that truly touches the ball has
//     |p_computed| <= R + delta with delta^2 <= 3*256 u^2 (|C|^2+|o|^2+|oc|^2) = 2.7e-12 (...), and
//     (R + delta)^2 <= 1.1 R^2 + 11 delta^2 <= 1.1 R^2 + 3e-11 (...);  |oc|^2 <= 2|C|^2 + 2|o|^2;
//   * a line whose world distance from C exceeds sqrt(1.1) R misses the object-space ball by >= 10 % of
//     ext^2 in the reference's discriminant, whose FP64 rounding error is <= ~1e3 * 2^-53 * kappa^2 *
//     (|C|^2+|o|^2+|oc|^2)/R^2 relative to it (kappa = cond(M)); shapes with kappa > 30 are never culled,
//     which keeps that term below 1e-10 (...) as well;
//   * B = 2e-10 >= 3e-11 + 1e-10;
//   * NaN / Inf operands make the comparisons false -> the exact test runs.
// Rectangles are never culled: a ray lying in their plane gives t = NaN, which the reference accepts
// (SURVEY A.6), whatever its distance from the rectangle.  Ray-marched shapes are handled by march_needed.
// Evidence: RT_ISECT_VERIFY runs the literal loop beside the culled one on every ray and tests every
// culled (ray, shape) pair exactly; tests/test_gpu_intersect.py requires zero disagreements.
//
// Hierarchy (CullTree).  Testing ~490 leaf balls per segment made k_extend FP32-issue bound, so the leaf
// balls sit under two levels of bounding balls: the culled shapes are clustered spatially (median
// splits) into GROUPS of <= 16, every 32 consecutive groups share a ROOT.  A lane tests the roots, the 32
// group balls under each root its line touches, the 16 leaf balls under each group it touches, and runs
// the exact FP64 test on the surviving leaves.  The visiting order is no longer the shape order; the
// sequential loop's "later shape wins ties" is applied explicitly (analytic_test).  Shapes that are
// never culled (Rectangles, ill-conditioned transforms), whose ball is much larger than the typical one
// (ground spheres) or scenes too small to be worth a tree go to a FLAT list tested as before.
// A node ball (c, Rn) encloses every member ball: Rn >= |C_i - c| + R_i.  It is rejected iff
//     |p|^2 > An + 101 * 3B |o|^2,    An = 1.01 (s Rn + sqrt(3B) (|c| + Rn))^2,  s = sqrt(1.1),
// which implies the member's own (exact-arithmetic) rejection with the FP64 slack it needs:
//   * (x + y)^2 <= 1.01 x^2 + 101 y^2, so rejection means |p|_computed > s Rn + sqrt(3B)(|c| + Rn + |o|);
//   * the FP32 error of |p| is delta <= 28u * 2(|c| + |o|) = 3.3e-6 (|c| + |o|) < (sqrt(3B) - sqrt(3e-10))(...),
//     so the true distance D of the line from c exceeds s Rn + sqrt(E), E = 3e-10 ((|c| + Rn)^2 + |o|^2)
//     >= the member's FP64 slack 3e-10 (|C_i|^2 + |o|^2);
//   * the distance from C_i is >= D - |C_i - c| > s R_i + (s - 1)|C_i - c| + sqrt(E) >= s R_i + sqrt(E),
//     i.e. d_i^2 > 1.1 R_i^2 + E: exactly what the leaf test certifies.  c is chosen FP32-representable.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#include "../../include/rt_b200.h"

namespace rt {

#define RT_CULL_B 2e-10
#define RT_CULL_MAX_KAPPA 30.0

// ---- host: one table entry per shape --------------------------------------------------------------
// (cx, cy, cz, A): A = 1.1 R^2 + 3B|C|^2 rounded up; A = +inf: never culled; A = -inf: never tested
// (padding and ray-marched shapes, masked out by the chunk's valid bits anyway).
// `ext`: object-space radius of the shape's bounding ball where the kind alone does not tell (Torus: radius + tube_radius).
inline float4 cull_entry(const double* m, int kind, double* radius_out = nullptr, double ext = 0.0) {
    if (radius_out) *radius_out = INFINITY;
    const float INF = INFINITY;
    float4 never = make_float4(0.f, 0.f, 0.f, INF);
    if (kind == RT_SHAPE_MARCH) return make_float4(0.f, 0.f, 0.f, -INF);
    if (kind == RT_SHAPE_TORUS && !(ext > 0.0 && ext < 1e150)) return never;
    if (kind != RT_SHAPE_SPHERE && kind != RT_SHAPE_CUBE && kind != RT_SHAPE_TORUS) return never;
    const double a[3][3] = {{m[0], m[1], m[2]}, {m[4], m[5], m[6]}, {m[8], m[9], m[10]}};
    const double tv[3] = {m[3], m[7], m[11]};
    double c[3][3];  // cofactors
    c[0][0] = a[1][1] * a[2][2] - a[1][2] * a[2][1];
    c[0][1] = a[1][2] * a[2][0] - a[1][0] * a[2][2];
    c[0][2] = a[1][0] * a[2][1] - a[1][1] * a[2][0];
    c[1][0] = a[0][2] * a[2][1] - a[0][1] * a[2][2];
    c[1][1] = a[0][0] * a[2][2] - a[0][2] * a[2][0];
    c[1][2] = a[0][1] * a[2][0] - a[0][0] * a[2][1];
    c[2][0] = a[0][1] * a[1][2] - a[0][2] * a[1][1];
    c[2][1] = a[0][2] * a[1][0] - a[0][0] * a[1][2];
    c[2][2] = a[0][0] * a[1][1] - a[0][1] * a[1][0];
    const double det = a[0][0] * c[0][0] + a[0][1] * c[0][1] + a[0][2] * c[0][2];
    if (!(fabs(det) > 0.0) || !isfinite(det)) return never;
    double inv[3][3];  // M^-1 = adj(M) / det, adj = cofactor^T
    for (int r = 0; r < 3; r++)
        for (int k = 0; k < 3; k++) inv[r][k] = c[k][r] / det;
    auto gersh = [](const double x[3][3]) {  // >= lambda_max(x^T x) = ||x||_2^2
        double g[3][3];
        for (int r = 0; r < 3; r++)
            for (int k = 0; k < 3; k++) g[r][k] = x[0][r] * x[0][k] + x[1][r] * x[1][k] + x[2][r] * x[2][k];
        double best = 0.0;
        for (int r = 0; r < 3; r++) best = fmax(best, fabs(g[r][0]) + fabs(g[r][1]) + fabs(g[r][2]));
        return best;
    };
    const double n_m = gersh(a), n_inv = gersh(inv);
    if (!isfinite(n_m) || !isfinite(n_inv)) return never;
    const double kappa = sqrt(n_m * n_inv);
    if (!(kappa <= RT_CULL_MAX_KAPPA)) return never;
    double C[3];
    for (int r = 0; r < 3; r++) C[r] = -(inv[r][0] * tv[0] + inv[r][1] * tv[1] + inv[r][2] * tv[2]);
    // Torus (shapes/mod.rs:429-452): a line whose distance from the centre exceeds radius + tube_radius has no real
    // intersection; the quartic's roots are then complex with imaginary parts of the order of the miss distance,
    // nowhere near the 1e-15 the reference accepts as real.  The ball test runs on the line like the Sphere's.
    const double ext2 = kind == RT_SHAPE_CUBE ? 3.0 : kind == RT_SHAPE_TORUS ? ext * ext : 1.0;
    const double R2 = ext2 * n_inv * (1.0 + 1e-9);
    const double cc = C[0] * C[0] + C[1] * C[1] + C[2] * C[2];
    const double A = 1.1 * R2 + 3.0 * RT_CULL_B * cc;
    if (!isfinite(A) || !isfinite(C[0]) || !isfinite(C[1]) || !isfinite(C[2])) return never;
    float Af = (float)A;
    if ((double)Af < A) Af = nextafterf(Af, INF);
    if (radius_out) *radius_out = sqrt(R2);
    return make_float4((float)C[0], (float)C[1], (float)C[2], Af);
}

// Bound of a ray-marched shape (ShapeFunction::intersect_bound, ray_marching.rs:135-145, 213-225): the
// reference solves the unit-sphere quadratic on o / radius, d / radius, i.e. a Sphere test with the inverse
// rows scaled by 1 / radius (componentwise for the Heart's ellipsoid).  A negative discriminant there means
// None for every max_t, so the same entry as for a Sphere applies (march_needed is skipped when the line
// misses the ball).  `radius`: the three object-space radii.
inline float4 cull_entry_march_bound(const double* m, const double radius[3]) {
    double ms[12];
    for (int r = 0; r < 3; r++)
        for (int k = 0; k < 4; k++) ms[4 * r + k] = m[4 * r + k] / radius[r];
    return cull_entry(ms, RT_SHAPE_SPHERE);
}

// ---- host: the two-level tree over the leaf entries -------------------------------------------------
#define RT_CULL_GROUP 16        // leaves per group
#define RT_CULL_ROOT_FANOUT 32  // groups per root
#define RT_CULL_NODE_RAY 101.0  // node tests use rhs = An + 101 * 3B |o|^2
#define RT_CULL_UPPER_MAX 4     // levels above the roots: each node covers 32 nodes of the level below
#define RT_CULL_TOP_TARGET 8    // levels are added until the top one has at most this many nodes

struct CullBall {
    double c[3], r;
};

struct CullTree {
    // table = [roots: n_roots][groups: n_groups (multiple of 8)][leaves: 16 * n_groups][flat: n_flat (multiple of 8)]
    std::vector<float4> table;
    std::vector<int> ids;       // [16 * n_groups + n_flat] shape index of every leaf / flat slot, -1 = padding
    std::vector<int> group_of;  // [n_shapes] group of a shape, -1 = flat list, -2 = not in the analytic loop
    std::vector<float4> leaf;   // [n_shapes] the shape's own entry (RT_ISECT_VERIFY)
    int n_roots = 0, n_groups = 0, n_flat = 0, n_flat_real = 0;
    std::vector<double> group_radius;  // [groups built] the FP64 radius each group entry was made from (rt_cull_tree_check)
    // ARBITRARY DEPTH: levels above the roots.  Level l (1-based) node i is a ball around the level l-1 nodes
    // [32 i, 32 i + 32) (level 0 = the roots), hence around every leaf ball below it -- the one property the
    // rejection proof above uses -- and is tested with the same node test.  upper = the levels' entries back to
    // back, level l at upper[upper_off[l]] with upper_count[l] entries; n_upper levels (0 for a scene of <= 8 roots,
    // i.e. up to ~4 000 shapes; 1 up to ~130 000; ...).  The walk tests a node when it reaches the first root of its
    // range and skips the whole range on rejection, so the roots tested per ray grow like log(n), not n / 512.
    int n_upper = 0, upper_off[RT_CULL_UPPER_MAX + 1] = {0, 0, 0, 0, 0}, upper_count[RT_CULL_UPPER_MAX + 1] = {0, 0, 0, 0, 0};
    std::vector<float4> upper;
    std::vector<CullBall> upper_ball;  // the FP64 balls the entries were made from (rt_cull_tree_check)
    std::vector<CullBall> root_ball;
    // the FP64 balls the leaf and group entries were made from, kept for the refit (rt_scene_update_transforms)
    std::vector<CullBall> leaf_ball;   // [n_shapes]
    std::vector<CullBall> group_ball;  // [groups built]
};

// One analytic shape's leaf entry and the FP64 ball the nodes above it must enclose: the entry's FP32-rounded centre
// with the radius padded by that rounding.  `inverse12`: its inverse rows; `params8`: its params row (may be null:
// a Torus is then never culled).  A non-finite radius means never culled (the entry has A = +inf).
inline float4 cull_leaf(const double* inverse12, int kind, const double* params8, bool no_cull, CullBall* ball) {
    double r;
    const double ext = (kind == RT_SHAPE_TORUS && params8) ? fabs(params8[0]) + fabs(params8[1]) : 0.0;
    float4 e = cull_entry(inverse12, kind, &r, ext);
    if (no_cull) e.w = INFINITY;
    *ball = CullBall{{(double)e.x, (double)e.y, (double)e.z}, r};
    if (isfinite(r)) {
        double cn = fabs(ball->c[0]) + fabs(ball->c[1]) + fabs(ball->c[2]);
        ball->r = r + cn * 1.2e-7;
    }
    return e;
}

// ball around member balls, FP32-representable centre
inline CullBall cull_enclose(const std::vector<CullBall>& m) {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (const CullBall& b : m)
        for (int k = 0; k < 3; k++) {
            lo[k] = fmin(lo[k], b.c[k] - b.r);
            hi[k] = fmax(hi[k], b.c[k] + b.r);
        }
    CullBall n;
    for (int k = 0; k < 3; k++) n.c[k] = (double)(float)(0.5 * (lo[k] + hi[k]));
    n.r = 0.0;
    for (const CullBall& b : m) {
        double dx = b.c[0] - n.c[0], dy = b.c[1] - n.c[1], dz = b.c[2] - n.c[2];
        n.r = fmax(n.r, sqrt(dx * dx + dy * dy + dz * dz) * (1.0 + 1e-12) + b.r);
    }
    n.r *= 1.0 + 1e-9;
    return n;
}

inline float4 cull_node_entry(const CullBall& n) {
    const double s = sqrt(1.1) * (1.0 + 1e-12);
    const double cn = sqrt(n.c[0] * n.c[0] + n.c[1] * n.c[1] + n.c[2] * n.c[2]);
    const double x = s * n.r + sqrt(3.0 * RT_CULL_B) * (cn + n.r);
    const double A = 1.0101 * x * x;  // 1.01 for the inequality above, the rest for the FP32 roundings of An + rhs
    if (!isfinite(A)) return make_float4(0.f, 0.f, 0.f, INFINITY);
    float Af = (float)A;
    if ((double)Af < A) Af = nextafterf(Af, INFINITY);
    return make_float4((float)n.c[0], (float)n.c[1], (float)n.c[2], Af);
}

// `inverse`: [n][12] inverse rows, `kind`: [n].  no_cull: every analytic shape goes to the flat list with
// A = +inf (debug switch RT_B200_NO_CULL); no_tree: flat list only (RT_B200_NO_CULL_TREE).
// `params`: [n][RT_SHAPE_PARAMS] (may be null: Torus shapes are then never culled).
inline CullTree cull_build(const double* inverse, const uint8_t* kind, int n, bool no_cull, bool no_tree,
                           const double* params = nullptr) {
    const float4 pad = make_float4(0.f, 0.f, 0.f, -INFINITY);
    CullTree t;
    t.group_of.assign(n, -2);
    t.leaf.assign(n, pad);
    std::vector<CullBall> ball(n);
    std::vector<int> tree, flat;
    std::vector<double> radii;
    for (int i = 0; i < n; i++) {
        if (kind[i] == RT_SHAPE_MARCH) continue;
        // the leaf entry's centre is the FP32-rounded one; the enclosing balls must contain the true ball:
        // cull_leaf pads the radius by the rounding of the centre
        t.leaf[i] = cull_leaf(inverse + (size_t)12 * i, kind[i], params ? params + (size_t)RT_SHAPE_PARAMS * i : nullptr,
                              no_cull, &ball[i]);
        if (isfinite(ball[i].r)) radii.push_back(ball[i].r);
    }
    double typical = 0.0;
    if (!radii.empty()) {
        std::nth_element(radii.begin(), radii.begin() + radii.size() / 2, radii.end());
        typical = radii[radii.size() / 2];
    }
    for (int i = 0; i < n; i++) {
        if (kind[i] == RT_SHAPE_MARCH) continue;
        const bool finite = isfinite(t.leaf[i].w) && isfinite(ball[i].r);
        if (no_tree || !finite || ball[i].r > 8.0 * typical) flat.push_back(i);
        else tree.push_back(i);
    }
    if ((int)tree.size() < 4 * RT_CULL_GROUP) {  // not worth a tree
        flat.insert(flat.end(), tree.begin(), tree.end());
        std::sort(flat.begin(), flat.end());
        tree.clear();
    }
    // spatial clustering: median split along the widest axis of the centres; the left part takes a whole
    // number of groups so that groups come out full
    std::vector<std::vector<int>> groups;
    struct Rec {
        static void split(std::vector<int> ids, const std::vector<CullBall>& ball, std::vector<std::vector<int>>& out) {
            if ((int)ids.size() <= RT_CULL_GROUP) {
                if (!ids.empty()) out.push_back(ids);
                return;
            }
            double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
            for (int i : ids)
                for (int k = 0; k < 3; k++) {
                    lo[k] = fmin(lo[k], ball[i].c[k]);
                    hi[k] = fmax(hi[k], ball[i].c[k]);
                }
            int ax = 0;
            if (hi[1] - lo[1] > hi[ax] - lo[ax]) ax = 1;
            if (hi[2] - lo[2] > hi[ax] - lo[ax]) ax = 2;
            std::stable_sort(ids.begin(), ids.end(), [&](int a, int b) { return ball[a].c[ax] < ball[b].c[ax]; });
            size_t n_groups = (ids.size() + RT_CULL_GROUP - 1) / RT_CULL_GROUP;
            size_t left = (n_groups / 2) * RT_CULL_GROUP;
            split(std::vector<int>(ids.begin(), ids.begin() + left), ball, out);
            split(std::vector<int>(ids.begin() + left, ids.end()), ball, out);
        }
    };
    Rec::split(tree, ball, groups);
    t.n_groups = (int)((groups.size() + 7) / 8 * 8);
    t.n_roots = (t.n_groups + RT_CULL_ROOT_FANOUT - 1) / RT_CULL_ROOT_FANOUT;
    t.n_flat_real = (int)flat.size();
    t.n_flat = (int)((flat.size() + 7) / 8 * 8);
    t.table.assign((size_t)t.n_roots + t.n_groups + (size_t)RT_CULL_GROUP * t.n_groups + t.n_flat, pad);
    t.ids.assign((size_t)RT_CULL_GROUP * t.n_groups + t.n_flat, -1);
    float4* roots = t.table.data();
    float4* grp = roots + t.n_roots;
    float4* leaves = grp + t.n_groups;
    float4* fl = leaves + (size_t)RT_CULL_GROUP * t.n_groups;
    std::vector<CullBall> gball(groups.size());
    for (size_t g = 0; g < groups.size(); g++) {
        std::vector<CullBall> m;
        std::sort(groups[g].begin(), groups[g].end());
        for (size_t k = 0; k < groups[g].size(); k++) {
            const int i = groups[g][k];
            m.push_back(ball[i]);
            leaves[g * RT_CULL_GROUP + k] = t.leaf[i];
            t.ids[g * RT_CULL_GROUP + k] = i;
            t.group_of[i] = (int)g;
        }
        gball[g] = cull_enclose(m);
        grp[g] = cull_node_entry(gball[g]);
        t.group_radius.push_back(gball[g].r);
    }
    t.leaf_ball = ball;
    t.group_ball = gball;
    t.root_ball.assign(t.n_roots, CullBall{{0.0, 0.0, 0.0}, -1.0});
    for (int r = 0; r < t.n_roots; r++) {
        std::vector<CullBall> m;
        for (size_t g = (size_t)r * RT_CULL_ROOT_FANOUT; g < std::min(groups.size(), (size_t)(r + 1) * RT_CULL_ROOT_FANOUT); g++)
            m.push_back(gball[g]);
        if (m.empty()) {
            roots[r] = pad;
            continue;
        }
        t.root_ball[r] = cull_enclose(m);
        roots[r] = cull_node_entry(t.root_ball[r]);
    }
    // levels above the roots (consecutive roots are spatial neighbours: the groups come out of the median splits in
    // order), until the top level is short
    {
        std::vector<CullBall> below = t.root_ball;
        while ((int)below.size() > RT_CULL_TOP_TARGET && t.n_upper < RT_CULL_UPPER_MAX) {
            const int lv = ++t.n_upper;
            const int count = ((int)below.size() + 31) / 32;
            t.upper_off[lv] = (int)t.upper.size();
            t.upper_count[lv] = count;
            std::vector<CullBall> here(count, CullBall{{0.0, 0.0, 0.0}, -1.0});
            for (int i = 0; i < count; i++) {
                std::vector<CullBall> m;
                for (int k = 32 * i; k < std::min(32 * i + 32, (int)below.size()); k++)
                    if (below[k].r >= 0.0) m.push_back(below[k]);
                if (m.empty()) {
                    t.upper.push_back(pad);
                } else {
                    here[i] = cull_enclose(m);
                    t.upper.push_back(cull_node_entry(here[i]));
                }
                t.upper_ball.push_back(here[i]);
            }
            below = here;
        }
    }
    for (size_t k = 0; k < flat.size(); k++) {
        fl[k] = t.leaf[flat[k]];
        t.ids[(size_t)RT_CULL_GROUP * t.n_groups + k] = flat[k];
        t.group_of[flat[k]] = -1;
    }
    return t;
}

// ---- device -----------------------------------------------------------------------------------------
struct CullRay {
    float ox, oy, oz, dx, dy, dz, rhs0, rhs1;  // rhs0 = 3B|o|^2 (leaf tests), rhs1 = 101 * 3B|o|^2 (node tests)
};

// FP32 operations of the pre-test, each rounded once (no contraction, no flush-to-zero): the _rn intrinsics on
// the device, the IEEE operations of the host compiler (-ffp-contract=off) in the host build that backs
// rt_cull_reached -- the same bits either way.
#ifdef __CUDA_ARCH__
#define RT_CF_FMA(a, b, c) __fmaf_rn(a, b, c)
#define RT_CF_MUL(a, b) __fmul_rn(a, b)
#define RT_CF_ADD(a, b) __fadd_rn(a, b)
#define RT_CF_SUB(a, b) __fsub_rn(a, b)
#define RT_CF_DIV(a, b) __fdiv_rn(a, b)
#define RT_CF_SQRT(a) __fsqrt_rn(a)
#define RT_CF_D2F(a) __double2float_rn(a)
#else
#define RT_CF_FMA(a, b, c) fmaf(a, b, c)
#define RT_CF_MUL(a, b) ((float)(a) * (float)(b))
#define RT_CF_ADD(a, b) ((float)(a) + (float)(b))
#define RT_CF_SUB(a, b) ((float)(a) - (float)(b))
#define RT_CF_DIV(a, b) ((float)(a) / (float)(b))
#define RT_CF_SQRT(a) sqrtf(a)
#define RT_CF_D2F(a) ((float)(a))
#endif

__host__ __device__ __forceinline__ CullRay make_cull_ray(double ox, double oy, double oz, double dx, double dy, double dz) {
    CullRay r;
    r.ox = RT_CF_D2F(ox);
    r.oy = RT_CF_D2F(oy);
    r.oz = RT_CF_D2F(oz);
    float x = RT_CF_D2F(dx), y = RT_CF_D2F(dy), z = RT_CF_D2F(dz);
    float s = RT_CF_FMA(z, z, RT_CF_FMA(y, y, RT_CF_MUL(x, x)));
    float inv = RT_CF_DIV(1.0f, RT_CF_SQRT(s));
    if (!(s > 1e-30f && s < 1e30f)) inv = NAN;  // zero / denormal / huge / NaN direction: nothing is culled
    r.dx = RT_CF_MUL(x, inv);
    r.dy = RT_CF_MUL(y, inv);
    r.dz = RT_CF_MUL(z, inv);
    float oo = RT_CF_FMA(r.oz, r.oz, RT_CF_FMA(r.oy, r.oy, RT_CF_MUL(r.ox, r.ox)));
    r.rhs0 = RT_CF_MUL((float)(3.0 * RT_CULL_B), oo);
    r.rhs1 = RT_CF_MUL((float)(RT_CULL_NODE_RAY * 3.0 * RT_CULL_B * (1.0 + 1e-6)), oo);
    return r;
}

// true: the exact test must run.  s = (C, A) from cull_entry.
__host__ __device__ __forceinline__ bool cull_pass(const CullRay& r, float4 s, float ray_rhs) {
    float ocx = RT_CF_SUB(s.x, r.ox), ocy = RT_CF_SUB(s.y, r.oy), ocz = RT_CF_SUB(s.z, r.oz);
    float b = RT_CF_FMA(ocz, r.dz, RT_CF_FMA(ocy, r.dy, RT_CF_MUL(ocx, r.dx)));
    float px = RT_CF_FMA(-b, r.dx, ocx), py = RT_CF_FMA(-b, r.dy, ocy), pz = RT_CF_FMA(-b, r.dz, ocz);
    float p2 = RT_CF_FMA(pz, pz, RT_CF_FMA(py, py, RT_CF_MUL(px, px)));
    float rhs = RT_CF_ADD(s.w, ray_rhs);
    return !(p2 > rhs);
}
__host__ __device__ __forceinline__ bool cull_pass(const CullRay& r, float4 s) { return cull_pass(r, s, r.rhs0); }
__host__ __device__ __forceinline__ bool cull_pass_node(const CullRay& r, float4 s) { return cull_pass(r, s, r.rhs1); }

}  // namespace rt
