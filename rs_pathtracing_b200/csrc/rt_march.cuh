// Exact-skip ray marching.
//
// RayMarchingShape::ray_intersect (src/world/shapes/ray_marching.rs:20-74) walks the ray in fixed
// steps of 0.01 in t — up to 23 925 strictly sequential iterations in cornell_box.json — looking for
// the first sign change of the surface polynomial, then refines it `depth` times with step *= -0.01.
// The candidate t it returns depends on every rounded partial sum of `t += step; p += step*dir`, so
// the loop cannot simply be replaced by a root finder.  This file reproduces its result BIT FOR BIT
// while executing a small fraction of the iterations.  Two independent facts make that possible:
//
//  (1) Skipping m steps of an accumulator exactly (advance_exact).  While a += s stays inside one
//      binade [2^e, 2^(e+1)), every step adds the SAME multiple D of ulp(a): the exact sum is
//      (T + S) ulp + rem with a constant remainder, so round-to-nearest always resolves it the same
//      way.  D is computed from the bit patterns of s and the binade, an exact tie is resolved by its
//      parity rule, and the steps that cross a binade boundary — the only ones whose rounding is
//      irregular — are executed literally.  m steps therefore cost O(number of binades crossed)
//      integer operations, and the result is the very double the reference's loop would hold.
//
//  (2) Proving that the skipped samples are uneventful (safe_extent).  Restricted to the ray the
//      surface function is a univariate polynomial g(tau) = f(p0 + tau d) of degree <= 6; its
//      coefficients are obtained once per ray by evaluating the same polynomial text on
//      degree-tracking polynomials (Poly<N>).  Starting from a point where |g| > M, hops of length
//          dtau = 2b / (|g'| + sqrt(g'^2 + 2 B2 b)),   b = |g| - M,   B2 >= max |g''| on the chord
//      stay inside {|g| >= M, same sign} by Taylor's theorem.  M bounds everything the
//      exact-arithmetic model ignores, with a 16-fold margin:
//        * the displacement of the accumulated sample against the model line p0 + tau d: MEASURED at
//          the current sample (e = p - (p0 + (t - t0) d)), plus at most half an ulp of t and of p per
//          future step for the m steps the jump may cover; seen through G >= sup |grad f| over the
//          marching region (march_bounds.hpp);
//        * the rounding of evaluating f (<= gamma_40 * F, F = the polynomial evaluated with absolute
//          values over the region, march_bounds.hpp) and of the model itself (1e-13 * sum |c_k| T^k).
//      On every skipped sample the reference's loop would therefore have found no sign change, no
//      |f| < 1e-15 and no range violation: it would only have executed `r = next`.
//
// After a skip the surface function is evaluated at the landing sample like the reference does
// (`r = next`) and compared with the polynomial's prediction; a mismatch (the model does not apply to
// this ray) restores the saved state and finishes the ray with the plain loop.  Wherever skipping is
// not worthwhile or not provable the reference's literal step is taken.
//
// The loop is written as a resumable state machine (Marcher::advance = one iteration of the
// reference's inner loop or one exact multi-step skip) so that k_march can hand a finished lane its next
// ray while the other lanes of the warp keep marching.
// tests/test_gpu_intersect.py compares t bit-exactly with the oracle for all six surfaces.
#pragma once
#include <cstring>

#include "rt_math.cuh"

namespace rt {

// ---- (1) exact multi-step advance ---------------------------------------------------------------
// advance_iter: one unit of progress (m > 0 on entry): a bounded literal walk near zero, or one binade --
// as many regular steps as provably stay inside it plus the few literal steps that cross its edge.
// advance_exact loops over it; k_march's cooperative advance interleaves it with other lanes' work.
// (host + device: the host build backs rt_advance_exact, which the CPU tests compare with the literal loop)
__host__ __device__ __forceinline__ long long adv_bits(double x) {
#ifdef __CUDA_ARCH__
    return __double_as_longlong(x);
#else
    long long r;
    memcpy(&r, &x, sizeof r);
    return r;
#endif
}
__host__ __device__ __forceinline__ double adv_from_bits(long long b) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double r;
    memcpy(&r, &b, sizeof r);
    return r;
#endif
}
// floor(num / D) for num < 2^52, D >= 1 -- or, when the quotient is 2^20 or more, a lower bound at least 3
// below it (any smaller value is safe: the remaining steps are simply handled by the next iterations).
// The quotient is estimated in FP32 (conversions + fast division: relative error < 2^-20, so the estimate
// is within 2 of the truth below 2^20) and corrected exactly with one 64-bit multiplication; the correction
// loops make the result independent of the quality of the estimate.  (__fdiv_rd is a subroutine call with a
// long slow path, a 64-bit integer division ~100 instructions.)
__host__ __device__ __forceinline__ long long adv_steps_to_edge(unsigned long long num, unsigned long long D) {
#ifdef __CUDA_ARCH__
    const float qf = __fdividef(__ull2float_rd(num), __ull2float_ru(D));
#else
    const float qf = (float)num / (float)D;
#endif
    if (!(qf < 1048576.0f)) {
        const long long room = (long long)(qf * 0.99999f) - 3;
        return room;
    }
    long long q = (long long)qf;
    long long r = (long long)num - q * (long long)D;  // |q D| < 2^21 * 2^52
    while (r < 0) {
        q--;
        r += (long long)D;
    }
    while (r >= (long long)D) {
        q++;
        r -= (long long)D;
    }
    return q;
}
__host__ __device__ __forceinline__ bool adv_mul_fits(unsigned long long a, unsigned long long b) {
#ifdef __CUDA_ARCH__
    return __umul64hi(a, b) == 0;
#else
    return (unsigned long long)(((unsigned __int128)a * b) >> 64) == 0;
#endif
}
__host__ __device__ __forceinline__ void advance_iter(double& a, const double s, long long& m) {
    const long long MANT = 0x000fffffffffffffLL;
    if (s == 0.0) {
        a = a + s;
        m = 0;
        return;
    }
    // Near zero (|a| < 32 |s|) a binade holds fewer than 32 steps: walking it literally (one DADD per step)
    // is cheaper than the per-binade bookkeeping below, and an accumulator that changes sign would
    // otherwise pay that bookkeeping for every binade between |s| and its starting magnitude, twice.
    const double near = 32.0 * fabs(s);
    if (fabs(a) < near) {
        // (literal steps are exact wherever they are taken: overshooting the zone by up to 3 of them is
        // harmless, so the test runs once per 4 steps)
#pragma unroll 1
        for (int c = 0; c < 4 && m >= 4 && fabs(a) < near; c++) {
            a = a + s;
            a = a + s;
            a = a + s;
            a = a + s;
            m -= 4;
        }
        if (m < 4) {
            while (m > 0 && fabs(a) < near) {
                a = a + s;
                m--;
            }
        }
        return;
    }
    const long long sb = adv_bits(fabs(s));
    const int sexp = (int)(sb >> 52);
    const long long Ms = (sb & MANT) | (1LL << 52);
    const bool s_neg = s < 0.0;
    const long long bits = adv_bits(a);
    const int exp = (int)((bits >> 52) & 0x7ff);
    const long long mant = bits & MANT;
    const bool a_neg = bits < 0;
    const int k = exp - sexp;           // ulp(a) = 2^k ulp(s):  s / ulp(a) = Ms / 2^k
    const bool up = (a_neg == s_neg);   // the magnitude grows
    // literal step wherever the regular-progression argument does not apply: zero / subnormal /
    // non-finite operands, a step comparable to the value itself, or the bottom of a binade
    // approached from above (the grid below it is finer)
    bool literal = exp == 0 || exp == 0x7ff || sexp == 0 || sexp == 0x7ff || k < 1 || (!up && mant == 0);
    long long D = 0;
    if (!literal && k <= 54) {
        const long long S = Ms >> k;
        const long long rem = Ms & ((1LL << k) - 1);
        const long long half = 1LL << (k - 1);
        if (rem > half) D = S + 1;
        else if (rem < half) D = S;
        else if (mant & 1) literal = true;   // exact tie from an odd mantissa: one literal step makes it even
        else D = S + (S & 1);                // exact tie from an even mantissa: round-half-even lands on even again
    }                                        // k > 54: |s| < ulp(a)/4, the sum rounds back to a (D = 0)
    if (literal) {
        a = a + s;
        m--;
        return;
    }
    if (D == 0) {  // a + s == a for every remaining step
        m = 0;
        return;
    }
    // Steps that stay inside this binade.  Going up, j steps are regular as long as mant + j D <= MANT: the
    // exact sum (mant + (j - 1) D + S) u + rem is below (MANT + 1) u = 2^(e+1), so it is rounded on this
    // binade's grid.  Going down, as long as mant - j D >= 1: the exact difference then lies above 2^e (by
    // u - rem > 0 when D = S + 1, by more than u / 2 when D = S).  So floor(num / D) steps are regular and
    // the one after them -- the only one whose rounding is irregular -- is taken literally.
    const unsigned long long num = (unsigned long long)(up ? (MANT - mant) : (mant - 1));
    const unsigned long long Du = (unsigned long long)D, mu = (unsigned long long)m;
    long long take;
    if (adv_mul_fits(mu, Du) && mu * Du <= num) {
        take = m;  // the whole jump stays inside the binade (the common case)
    } else {
        long long room = adv_steps_to_edge(num, Du);  // < m here (or a lower bound of it)
        if (room < 0) room = 0;
        take = room < m ? room : m;
    }
    if (take > 0) {
        a = adv_from_bits(up ? bits + take * D : bits - take * D);
        m -= take;
        if (m == 0) return;  // the common case: the whole jump in one binade
    }
    // at the binade edge: one literal step carries it across
    a = a + s;
    m--;
}

// returns the value `a` holds after m iterations of `a = a + s` in IEEE double arithmetic
__host__ __device__ __forceinline__ double advance_exact(double a, double s, long long m) {
    while (m > 0) advance_iter(a, s, m);
    return a;
}

// ---- (2) the surface function along the ray as a univariate polynomial ---------------------------
// Degree-tracking polynomial in tau: the product of a Poly<A> and a Poly<B> is a Poly<A+B>, so
// expanding a surface of degree 6 costs ~80 FMAs instead of the ~300 of a fixed-size truncated series.
template <int N>
struct Poly {
    static constexpr int degree = N;
    double c[N + 1];
};
template <int A, int B>
__host__ __device__ __forceinline__ Poly<A + B> operator*(const Poly<A>& a, const Poly<B>& b) {
    Poly<A + B> r;
#pragma unroll
    for (int k = 0; k <= A + B; k++) {
        double s = 0.0;
#pragma unroll
        for (int i = 0; i <= A; i++)
            if (k - i >= 0 && k - i <= B) s = fma(a.c[i], b.c[k - i], s);
        r.c[k] = s;
    }
    return r;
}
template <int A, int B>
__host__ __device__ __forceinline__ Poly<(A > B ? A : B)> operator+(const Poly<A>& a, const Poly<B>& b) {
    Poly<(A > B ? A : B)> r;
#pragma unroll
    for (int k = 0; k <= (A > B ? A : B); k++) r.c[k] = (k <= A ? a.c[k] : 0.0) + (k <= B ? b.c[k] : 0.0);
    return r;
}
template <int A, int B>
__host__ __device__ __forceinline__ Poly<(A > B ? A : B)> operator-(const Poly<A>& a, const Poly<B>& b) {
    Poly<(A > B ? A : B)> r;
#pragma unroll
    for (int k = 0; k <= (A > B ? A : B); k++) r.c[k] = (k <= A ? a.c[k] : 0.0) - (k <= B ? b.c[k] : 0.0);
    return r;
}
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator+(Poly<A> a, double b) { a.c[0] += b; return a; }
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator-(Poly<A> a, double b) { a.c[0] -= b; return a; }
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator+(double a, Poly<A> b) { b.c[0] += a; return b; }
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator-(double a, Poly<A> b) {
#pragma unroll
    for (int i = 0; i <= A; i++) b.c[i] = -b.c[i];
    b.c[0] += a;
    return b;
}
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator*(Poly<A> a, double b) {
#pragma unroll
    for (int i = 0; i <= A; i++) a.c[i] *= b;
    return a;
}
template <int A>
__host__ __device__ __forceinline__ Poly<A> operator*(double a, Poly<A> b) { return b * a; }
__host__ __device__ __forceinline__ Poly<1> poly_lin(double v, double d) {
    Poly<1> r;
    r.c[0] = v;
    r.c[1] = d;
    return r;
}

// degree of the surface polynomial along a ray
template <int KIND>
struct SurfDeg {
    static constexpr int value = (KIND == RT_SURF_DUPIN || KIND == RT_SURF_CUSHION) ? 4 : 6;
};

template <int DEG>
struct RayPoly {
    double c[DEG + 1];  // g(tau) = sum c[k] tau^k, tau = t - t0
    double t0;          // the value t had at the expansion point ...
    D3 p0;              // ... and the sample position there: the model line is p0 + tau d
    double tau_hi;      // the model covers tau in [0, tau_hi]
    double err0;        // evaluation / model rounding term of M
    double drift1;      // displacement bound per future step, already multiplied by the safety factor and G
};

#define RT_MARCH_SAFETY 16.0

// double -> float rounded towards +inf / -inf (the hop lengths are lower bounds: FP32, rounded to the safe side).  The
// host forms give the same floats, so the host build of the marcher (rt_march_candidates_host) plans the same jumps.
__host__ __device__ __forceinline__ float d2f_ru(double x) {
#ifdef __CUDA_ARCH__
    return __double2float_ru(x);
#else
    float f = (float)x;
    if ((double)f < x) f = nextafterf(f, INFINITY);
    return f;
#endif
}
__host__ __device__ __forceinline__ float d2f_rd(double x) {
#ifdef __CUDA_ARCH__
    return __double2float_rd(x);
#else
    float f = (float)x;
    if ((double)f > x) f = nextafterf(f, -INFINITY);
    return f;
#endif
}

// magnitude arithmetic (march_bounds.hpp's Mag, device side): every operation returns an upper bound of the sum of the
// absolute values of the terms it combines, so evaluating the surface polynomial's text on it bounds the
// "absolute-value polynomial" at the given |coordinates| -- and anywhere closer to the origin, componentwise.
struct MagD {
    double v;
};
__host__ __device__ __forceinline__ MagD operator+(MagD a, MagD b) { return MagD{a.v + b.v}; }
__host__ __device__ __forceinline__ MagD operator-(MagD a, MagD b) { return MagD{a.v + b.v}; }
__host__ __device__ __forceinline__ MagD operator*(MagD a, MagD b) { return MagD{a.v * b.v}; }
__host__ __device__ __forceinline__ MagD operator+(MagD a, double b) { return MagD{a.v + fabs(b)}; }
__host__ __device__ __forceinline__ MagD operator-(MagD a, double b) { return MagD{a.v + fabs(b)}; }
__host__ __device__ __forceinline__ MagD operator*(MagD a, double b) { return MagD{a.v * fabs(b)}; }
__host__ __device__ __forceinline__ MagD operator+(double a, MagD b) { return MagD{fabs(a) + b.v}; }
__host__ __device__ __forceinline__ MagD operator-(double a, MagD b) { return MagD{fabs(a) + b.v}; }
__host__ __device__ __forceinline__ MagD operator*(double a, MagD b) { return MagD{fabs(a) * b.v}; }

// expansion of f along the ray around the current sample (t, p); the model must cover tau in [0, tau_hi]
template <int KIND>
__host__ __device__ __forceinline__ void expand_ray(const double* q, D3 p, D3 d, double t, double t_end, double tau_hi,
                                           double G, double F, RayPoly<SurfDeg<KIND>::value>& P) {
    constexpr int DEG = SurfDeg<KIND>::value;
    auto g = surface_func_t<KIND>(q, poly_lin(p.x, d.x), poly_lin(p.y, d.y), poly_lin(p.z, d.z));
    static_assert(decltype(g)::degree == DEG, "SurfDeg out of date");
    double scale = 0.0;
    double pw = 1.0;  // tau_hi^k
#pragma unroll
    for (int k = 0; k <= DEG; k++) {
        P.c[k] = g.c[k];
        scale += fabs(g.c[k]) * pw;
        pw *= tau_hi;
    }
    const double EPS = 1.1102230246251565e-16;  // 2^-53: half an ulp, relative
    const double tmax = fmax(fabs(t), fabs(t_end)) + tau_hi;
    const double dmax = fmax(fmax(fabs(d.x), fabs(d.y)), fabs(d.z));
    const double pmax = fmax(fmax(fabs(p.x), fabs(p.y)), fabs(p.z)) + tau_hi * dmax;
    const double dlen = fabs(d.x) + fabs(d.y) + fabs(d.z);  // >= |d|
    // one step moves the sample off the model line by at most half an ulp of p per component, half an ulp
    // of t along d, and the rounding of `step * dir` (relative 2^-53 of one step, far below the former)
    const double per_step = EPS * (2.0 * pmax + tmax * dlen);
    P.t0 = t;
    P.p0 = p;
    P.tau_hi = tau_hi;
    P.drift1 = RT_MARCH_SAFETY * G * per_step;
    // rounding of f (gamma_n F with n ~ 40 operations -> 4.4e-15 F), of the model's coefficients and of
    // its Horner evaluation / Taylor shift (a few 1e-16 * scale), of measuring e (8 steps' worth)
    P.err0 = RT_MARCH_SAFETY * (1e-14 * F + 1e-14 * scale) + 8.0 * P.drift1 + 1e-300;
}


// ---- (3) a ray that provably never comes near the surface: None without marching ----------------------------
// Two thirds of the marched rays of cornell_box cross the Heart's bounding ellipsoid without touching the Heart.
// For them the reference executes `r = next` thousands of times and leaves through the range check; the exact
// values of t and p never matter.  If sigma g(tau) > M(tau) on the WHOLE stretch the samples can fall on -- tau up to
// (end - t0) + 3 step: the last sample evaluated is the first one with t > end -- then no sample sees a sign change
// or |f| < 1e-15 (the argument of (2), with the a-priori displacement bound of tau / step steps at the sample at
// tau), and the result is None.  M(tau) is linear in tau, so sigma g - M is a polynomial of the same degree, and the
// proof is the convex-hull property of its Bernstein form: on [a, b], min_i b_i <= p <= max_i b_i, b = the Bernstein
// coefficients of p over [a, b]; the hull is tightened by de Casteljau subdivision at the midpoint (two levels: 93 %
// of the misses among random chords of the Heart's bound, against 52 % for the undivided hull).  Marcher::begin has
// the details (the interval starts half a step in; the value at sample 0 only lends its sign).  Straight-line code:
// k_march_filter runs it for every queued (ray, shape) pair with full warps, before the marcher sees the queue.
// Rounding: the conversion and each subdivision level are convex combinations / binomial sums of <= 7 terms bounded
// by scale = sum |c_k| L^k, error <= 3e-15 scale in total; err0 >= 1.6e-13 scale is subtracted once more for it.
template <int DEG>
__host__ __device__ __forceinline__ bool bern_hull_clear(const double (&b)[DEG + 1], double thr, bool positive) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i <= DEG; i++) ok = ok && (positive ? b[i] > thr : b[i] < -thr);   // NaN -> false
    return ok;
}
template <int DEG>
__host__ __device__ __forceinline__ void bern_split(const double (&b)[DEG + 1], double (&l)[DEG + 1], double (&r)[DEG + 1]) {
    double w[DEG + 1];
#pragma unroll
    for (int i = 0; i <= DEG; i++) w[i] = b[i];
#pragma unroll
    for (int j = 0; j <= DEG; j++) {
        l[j] = w[0];
        r[DEG - j] = w[DEG - j];
#pragma unroll
        for (int i = 0; i < DEG - j; i++) w[i] = 0.5 * (w[i] + w[i + 1]);
    }
}
// true: |g(tau)| > thr with the sign of c[0] for every tau in [0, L]
template <int DEG>
// (host + device: the host build backs rt_bernstein_clear, which the CPU tests compare with dense sampling)
__host__ __device__ __forceinline__ bool bernstein_clear(const double (&c)[DEG + 1], double L, double thr) {
    static_assert(DEG == 4 || DEG == 6, "binomial table");
    double b[DEG + 1];
    double pw = 1.0;
#pragma unroll
    for (int k = 0; k <= DEG; k++) {
        // 1 / C(DEG, k)
        const double inv_binom = DEG == 6 ? (k == 0 || k == 6 ? 1.0 : k == 1 || k == 5 ? 1.0 / 6.0 : k == 2 || k == 4 ? 1.0 / 15.0 : 1.0 / 20.0)
                                          : (k == 0 || k == 4 ? 1.0 : k == 2 ? 1.0 / 6.0 : 0.25);
        b[k] = c[k] * pw * inv_binom;
        pw *= L;
    }
    // b_i = sum_k C(i, k) a_k / C(DEG, k): the binomial transform, by Pascal's rule
#pragma unroll
    for (int j = 1; j <= DEG; j++)
#pragma unroll
        for (int i = DEG; i >= j; i--) b[i] += b[i - 1];
    const bool positive = b[0] > 0.0;
    // the end values are values of g itself: no subdivision helps when they fail
    if (!(positive ? (b[0] > thr && b[DEG] > thr) : (b[0] < -thr && b[DEG] < -thr))) return false;
    if (bern_hull_clear<DEG>(b, thr, positive)) return true;
    double l[DEG + 1], r[DEG + 1];
    bern_split<DEG>(b, l, r);
    bool ok = true;
    {
        if (!bern_hull_clear<DEG>(l, thr, positive)) {
            double ll[DEG + 1], lr[DEG + 1];
            bern_split<DEG>(l, ll, lr);
            ok = bern_hull_clear<DEG>(ll, thr, positive) && bern_hull_clear<DEG>(lr, thr, positive);
        }
    }
    if (ok && !bern_hull_clear<DEG>(r, thr, positive)) {
        double rl[DEG + 1], rr[DEG + 1];
        bern_split<DEG>(r, rl, rr);
        ok = bern_hull_clear<DEG>(rl, thr, positive) && bern_hull_clear<DEG>(rr, thr, positive);
    }
    return ok;
}

#define RT_MARCH_MIN_JUMP 8
#ifndef RT_MARCH_LAND_COOLDOWN
#define RT_MARCH_LAND_COOLDOWN 6
#endif
enum { RT_MARCH_MORE = 0, RT_MARCH_DONE = 1, RT_MARCH_MISS = 2 };
enum { RT_PHASE_END = 0, RT_PHASE_ATTEMPT = 1, RT_PHASE_LITERAL = 2 };

// RayMarchingShape::ray_intersect's loops (ray_marching.rs:27-57) as a resumable state machine.
// G / F = gradient and magnitude bounds of the surface over its marching region; a non-finite bound
// (or a chord of few steps) gives exactly the plain loop.
//
// One iteration of the reference's inner loop is  [range check]  then either
//   attempt():  try to replace the next m >= RT_MARCH_MIN_JUMP iterations by one exact jump, or
//   literal():  the reference's own step.
// phase() says which of the two the lane would do next; k_march lets a warp vote so that the expensive
// attempt runs with many lanes at once.
template <int KIND, bool PROF = false>
struct Marcher {
    static constexpr int DEG = SurfDeg<KIND>::value;
    unsigned prof[8];  // PROF only: literal steps at level 0 / at refinement levels, jumps, hops, misses proven by the
                       // Bernstein hull / by the hop loop, plans that found nothing to skip at level 0 / at a refinement level
    const double* q;
    D3 d;
    double start, end, G, F;
    // the reference's loop state
    double t, r, step;
    D3 p, sd;
    int it, depth;
    unsigned long long n;  // surface evaluations (statistics, and the spin guard)
    // skip machinery
    double step0;
    bool skip_ok;
    bool local_model;    // P is the model re-expanded around the level-0 crossing (refine_model)
    int cooldown, backoff;
    RayPoly<DEG> P;

    // hull: try the miss proof (3) right away (off when k_march_filter has already tried it for this ray)
    __host__ __device__ __forceinline__ void begin(const double* q_, D3 o_, D3 d_, double start_, double end_, double G_,
                                          double F_, bool hull = true) {
        q = q_; d = d_; start = start_; end = end_; G = G_; F = F_;
        step = q[1];
        step0 = step;
        depth = (int)q[2];
        t = start;
        p = o_ + t * d;
        r = surface_func<KIND>(q, p);
        n = 0;
        it = 0;
        sd = step * d;  // `step * dir`, loop-invariant until the step changes
        cooldown = 0;
        backoff = 4;
        if (PROF) prof[0] = prof[1] = prof[2] = prof[3] = prof[4] = prof[5] = prof[6] = prof[7] = 0;
        // skipping pays when the chord holds many steps (NaN-proof comparisons)
        skip_ok = (G == G) && G < 1e300 && (F == F) && F < 1e300 && step > 0.0 && (end - start) > 64.0 * step &&
                  (end - start) < 1e300;
        local_model = false;
        if (skip_ok) {
            // the model along the ray, expanded around the first sample; covers every later sample of the ray
            expand_ray<KIND>(q, p, d, t, end, (end - t) + 4.0 * step0, G, F, P);
            n += 2;  // cost of the expansion in evaluation-equivalents (statistics only)
#ifndef RT_MARCH_NO_MISS_PROOF
            // (3): no sample of this ray can see an event -> None.  The samples the loop TESTS are n = 1, 2, ... (the
            // first one only lends its sign to the comparison with the second), sample n sits at tau_n = t_n - t0 with
            // n <= tau_n / step + 1, and its displacement from the model line is at most n steps' worth (e = 0 at the
            // expansion sample): M(tau) = err0 + (tau / step + 4) drift1 bounds what the model ignores AT that sample.
            // So it suffices that  sigma g(tau) - M(tau) > 0  on [step / 2, L] -- a polynomial of the same degree, the
            // band being linear in tau -- and that r, the value at sample 0, is not of the opposite sign.  Starting
            // half a step in matters: a ray that leaves the surface it was scattered from has |g(0)| ~ 1e-9, far
            // inside the band of a 20 000-step chord, but is 1e-4 away from zero one step later.
            const double L = miss_span(t);
            // (depth 0: the reference runs no loop at all and returns the hit at t = start, whatever the surface does)
            if (hull && depth > 0 && miss_drift_ok(L)) {
                const double ta = 0.5 * step0;
                double sh[DEG + 1];
#pragma unroll
                for (int k = 0; k <= DEG; k++) sh[k] = P.c[k];
#pragma unroll
                for (int i = 0; i < DEG; i++)   // Taylor shift to ta: g(ta + x) = sum sh[k] x^k
#pragma unroll
                    for (int j = DEG - 1; j >= i; j--) sh[j] = fma(ta, sh[j + 1], sh[j]);
                const bool positive = sh[0] > 0.0;
                if (positive ? !(r < 0.0) : !(r > 0.0)) {
                    if (!positive) {
#pragma unroll
                        for (int k = 0; k <= DEG; k++) sh[k] = -sh[k];
                    }
                    // err0 twice: once for the band, once for the rounding of the shift and of the Bernstein form
                    sh[0] -= fmax(2.0 * P.err0 + (ta / step0 + 4.0) * P.drift1, 2e-15);   // (>= 2e-15: approx_equal's exit)
                    sh[1] -= P.drift1 / step0;
                    if (bernstein_clear<DEG>(sh, L - ta, 0.0)) {
                        t = INFINITY;   // phase() -> RT_PHASE_END, finish() -> RT_MARCH_MISS
                        if (PROF) prof[4]++;
                    }
                }
            }
#endif
        }
    }
    // the stretch of tau (from the sample at t_now, level 0) on which the remaining samples of the ray can fall: the
    // last one evaluated is the first with t > end, i.e. at most end + step (+ rounding); 3 steps for margin
    __host__ __device__ __forceinline__ double miss_span(double t_now) const { return (end - t_now) + 3.0 * step0; }
    // the accumulated t stays within half a step of t0 + n step for all the steps of the stretch (so that "the first
    // sample with t > end" is where the model says): n roundings of at most half an ulp of the largest t
    __host__ __device__ __forceinline__ bool miss_drift_ok(double L) const {
        const double tmax = fmax(fabs(start), fabs(end)) + 4.0 * step0;
        return (L / step0 + 4.0) * 1.1102230246251565e-16 * tmax < 0.25 * step0;
    }

    // what the next iteration starts with.  RT_PHASE_END: the loops are over (finish() tells how)
    __host__ __device__ __forceinline__ int phase() const {
        if (it >= depth) return RT_PHASE_END;
        // n > RT_MARCH_BUDGET: t + step == t (step underflowed against t); the reference would spin
        // forever, a kernel must not: report a miss
        if (t > end || t < start || n > RT_MARCH_BUDGET) return RT_PHASE_END;
        return (skip_ok && cooldown == 0) ? RT_PHASE_ATTEMPT : RT_PHASE_LITERAL;
    }
    // valid when phase() == RT_PHASE_END
    __host__ __device__ __forceinline__ int finish() const { return it >= depth ? RT_MARCH_DONE : RT_MARCH_MISS; }

    // Try one exact multi-step jump from the current sample.  Afterwards either the state is m
    // iterations further (the reference would have executed exactly `r = next` in each of them), or
    // nothing changed except cooldown / skip_ok, so that phase() now answers RT_PHASE_LITERAL.
    // The attempt is split in three so that k_march can run the middle part -- the exact advance of the
    // four accumulators t, p.x, p.y, p.z, whose loops over binades are the most divergent code of the
    // marcher -- cooperatively, one accumulator per lane (coop_advance in rt_march_kernels.cu):
    //   attempt_plan():  how many iterations m can provably be skipped (0: none; cooldown is set)
    //   [advance t, p by m steps exactly]
    //   attempt_land():  the reference's `r = next` at the landing sample + the model self-check
    struct Plan {
        double s[DEG + 1];  // the model shifted to the sample + `shift`: g(tau + shift + x) = sum s[k] x^k (x signed)
        double M;           // the uncertainty band of this jump (of its last stage)
        // state of the hop loop (plan_begin / plan_hop / plan_end)
        double shift;       // signed displacement of the expansion point of s[] from the current sample
        double sig, g, dg, span, abs_step, dir, span_limit, base;
        float B2;
        int hop, stage;
        double jump_limit;    // how far a jump may go (span_limit reaches further while a miss can still be proven)
        bool miss_possible;   // span_limit = the whole stretch the ray's remaining samples can fall on
        bool newton_limited;  // this stage's span was cut by the Newton-distance rule, not by the range limit
        bool more;            // stopped at the stage limit, not at the |g| = M boundary: attempt again after landing
    };
#define RT_MARCH_MAX_STAGES 6
    // attempt_plan = plan_begin, then plan_hop until it returns false, then plan_end.
    //
    // The hops are planned in STAGES.  A stage bounds |g''| over its whole span, so from far away the bound
    // is loose and the hops stall (or the span, limited to twice the Newton distance, ends) well before the
    // |g| = M boundary.  Re-planning from the point reached needs no exact advance -- only a Taylor shift
    // of the model (21 FMAs) and a new, tighter bound -- so it is done right here; the accumulators are
    // advanced once, by the total.  (It used to take a landing + a fresh attempt: 2.9 attempts per ray at
    // level 0, 1.4 of them failing.)  M grows from stage to stage with the number of steps the jump may then
    // cover; the stretch proven by an earlier stage only needed the smaller M of that stage.
    __host__ __device__ __forceinline__ void plan_stage(Plan& pl) {
        const double remaining = fmax(pl.span_limit - fabs(pl.shift), 0.0);
        // do not look further than twice the Newton distance to the next root: the |g''| bound grows with the span
        const double span = fmin(remaining, (2.0 * fabs(pl.s[0]) / fabs(pl.s[1]) + 32.0 * pl.abs_step));  // fmin ignores a NaN quotient
        pl.newton_limited = span < remaining;
        const double m_max = (fabs(pl.shift) + span) / pl.abs_step + 4.0;
        // (never below 2e-15: a skipped sample must also stay clear of the reference's `approx_equal(next, 0.0)` exit,
        // |f| < 1e-15, and for a surface of tiny magnitude the error terms alone would not guarantee that)
        pl.M = fmax(pl.base + m_max * P.drift1, 2e-15);
        // furthest sigma in [0, span] such that the whole stretch is provably inside {|g| >= M, same sign}:
        // hops of length 2b / (|g'| + sqrt(g'^2 + 2 B2 b)), b = |g| - M, B2 >= max |g''| over the span.
        // The hop length is a lower bound, so it is computed in FP32 (rounded toward safety, shortened 1 %).
        double b2 = 0.0, pw = 1.0;
#pragma unroll
        for (int k = 2; k <= DEG; k++) {
            b2 += (double)(k * (k - 1)) * fabs(pl.s[k]) * pw;
            pw *= span;
        }
        pl.B2 = d2f_ru(b2 * (1.0 + 1e-9));
        pl.sig = 0.0;
        pl.g = pl.s[0];
        pl.dg = pl.s[1];
        pl.span = span;
        pl.hop = 0;
    }
    // The refinement levels (it > 0) never leave the last level-0 step around the first sign change, but their steps
    // shrink to 1e-8: the band M has to be a fraction of ONE such step's change of g (~3e-10 on cornell_box's Heart)
    // for a jump to be provable.  The model expanded at the chord's start cannot deliver that: shifting it hundreds of
    // world units costs ~1e-16 * sum |c_k| tau^k of absolute accuracy (err0's `scale` term, 1e-9 and more), and the
    // evaluation term uses the magnitude bound F of the whole region.  Measured: 70 % of the hit rays walked the last
    // level literally (~50 steps) after an empty plan.  So the first plan of a refinement level re-expands f around
    // the current sample: centre half a window back (the model line only runs forward), window = 2 x 1.02 level-0
    // steps, F = the absolute-value polynomial at the window's largest |coordinates|.  P.p0 / P.t0 need not be
    // samples: plan_begin measures the displacement e of the real sample from the model line, whatever it is.
    __host__ __device__ __forceinline__ void refine_model() {
        const double h = 1.02 * step0;
        const D3 pc = mk(fma(-h, d.x, p.x), fma(-h, d.y, p.y), fma(-h, d.z, p.z));
        const double w = 2.0 * h;
        const MagD fm = surface_func_t<KIND, MagD>(q, MagD{fabs(pc.x) + w * fabs(d.x)}, MagD{fabs(pc.y) + w * fabs(d.y)},
                                                   MagD{fabs(pc.z) + w * fabs(d.z)});
        double f_loc = fm.v * (1.0 + 1e-9);
        if (!(f_loc < F)) f_loc = F;   // (NaN / inf: the region's bound)
        expand_ray<KIND>(q, pc, d, t - h, t + h, w, G, f_loc, P);
        n += 2;
        local_model = true;
    }
    __host__ __device__ __forceinline__ void plan_begin(Plan& pl) {
        double(&s)[DEG + 1] = pl.s;
        const double abs_step = fabs(step);
        const double dir = step > 0.0 ? 1.0 : -1.0;
        double tau = t - P.t0;
        // Taylor shift to the current sample: g(tau + sigma) = sum s[k] sigma^k
#pragma unroll
        for (int k = 0; k <= DEG; k++) s[k] = P.c[k];
#pragma unroll
        for (int i = 0; i < DEG; i++)
#pragma unroll
            for (int j = DEG - 1; j >= i; j--) s[j] = fma(tau, s[j + 1], s[j]);
#ifndef RT_MARCH_NO_LOCAL_MODEL
        if (it > 0 && !local_model) {
            // decided once per ray, at its first refinement plan: re-expand when the chord-wide model's own error
            // term is worth more than two of the FINEST steps (|g'| x step x 0.01^(depth - 1)) -- otherwise the last
            // level could never jump; a model that is already sharper than that (short chords, DupinCyclide under a
            // scale of 2) is kept, the re-expansion would only cost
            local_model = true;
            double finest = step0;
            for (int l = 1; l < depth; l++) finest *= 0.01;
            if (P.err0 > 2.0 * fabs(s[1]) * finest) {
                refine_model();
                tau = t - P.t0;
#pragma unroll
                for (int k = 0; k <= DEG; k++) s[k] = P.c[k];
#pragma unroll
                for (int i = 0; i < DEG; i++)
#pragma unroll
                    for (int j = DEG - 1; j >= i; j--) s[j] = fma(tau, s[j + 1], s[j]);
            }
        }
#endif
        // the range checks must not fire on skipped samples: stay 2 steps inside [start, end] and the model
        double tau_lim = (dir > 0.0 ? end : start) - P.t0 - dir * 2.0 * abs_step;
        tau_lim = fmin(fmax(tau_lim, 0.0), P.tau_hi);
        pl.span_limit = fmax((tau_lim - tau) * dir, 0.0);
        pl.jump_limit = pl.span_limit;
        pl.miss_possible = false;
#ifndef RT_MARCH_NO_MISS_PROOF
        // (3) again, from wherever the ray is at level 0: let the hops run on to the end of the stretch the remaining
        // samples can fall on; if they get there the ray is a miss and nothing has to be advanced
        if (it == 0 && dir > 0.0) {
            const double L = miss_span(t);
            if (tau + L <= P.tau_hi && miss_drift_ok(L)) {
                pl.span_limit = L;
                pl.miss_possible = true;
            }
        }
#endif
        // the part of M that does not depend on the length of the jump: the displacement of the sample
        // against the model line, measured now, and the evaluation / model rounding
        const double ex = p.x - fma(tau, d.x, P.p0.x), ey = p.y - fma(tau, d.y, P.p0.y),
                     ez = p.z - fma(tau, d.z, P.p0.z);
        pl.base = RT_MARCH_SAFETY * G * (fabs(ex) + fabs(ey) + fabs(ez)) + P.err0;
        pl.abs_step = abs_step;
        pl.dir = dir;
        pl.shift = 0.0;
        pl.stage = 0;
        pl.more = false;
        plan_stage(pl);
    }
    // the stage ended short of the |g| = M boundary: re-plan from the point reached, if that may help
    __host__ __device__ __forceinline__ bool plan_next_stage(Plan& pl, bool progressed) {
        if (!progressed) return false;
        if (pl.stage + 1 >= RT_MARCH_MAX_STAGES) {
            pl.more = true;
            return false;
        }
        const double x = pl.dir * pl.sig;
#pragma unroll
        for (int i = 0; i < DEG; i++)
#pragma unroll
            for (int j = DEG - 1; j >= i; j--) pl.s[j] = fma(x, pl.s[j + 1], pl.s[j]);
        pl.shift += x;
        pl.stage++;
        plan_stage(pl);
        return true;
    }
    // one hop; false when the planning is over
    __host__ __device__ __forceinline__ bool plan_hop(Plan& pl) {
        if (pl.hop >= 32) return plan_next_stage(pl, pl.sig > 0.0);
        pl.hop++;
        if (PROF) prof[3]++;
        const double b = fabs(pl.g) - pl.M;
        if (!(b > 0.0)) return false;  // at the boundary of the uncertainty band: the jump ends here
        const float bf = d2f_rd(b);
        const float af = d2f_ru(fabs(pl.dg));
        const float den = af + sqrtf(fmaf(af, af, 2.0f * pl.B2 * bf));
        const double dt = (double)(0.99f * (2.0f * bf / den));
        const double ns = pl.sig + dt;
        if (ns >= pl.span) {
            pl.sig = pl.span;
            if (pl.newton_limited) return plan_next_stage(pl, pl.sig > 0.0);
            return false;  // the range limit
        }
        if (!(dt > pl.abs_step)) return plan_next_stage(pl, pl.sig > 8.0 * pl.abs_step);  // stalled: loose |g''| bound?
        pl.sig = ns;
        const double x = pl.dir * pl.sig;
        double v = pl.s[DEG], dv = 0.0;
#pragma unroll
        for (int k = DEG - 1; k >= 0; k--) {
            dv = fma(dv, x, v);
            v = fma(v, x, pl.s[k]);
        }
        pl.g = v;
        pl.dg = dv;
        return true;
    }
    // the number of iterations that can be skipped (0: none, cooldown is set)
    __host__ __device__ __forceinline__ long long plan_end(const Plan& pl) {
        double reach = fabs(pl.shift) + pl.sig;
        if (pl.miss_possible) {
            // the last stage ran into the range limit (plan_hop: sig = span, not Newton-limited): proven to the end
            if (!pl.newton_limited && pl.sig >= pl.span && reach >= pl.span_limit * (1.0 - 1e-12)) {
                t = INFINITY;   // phase() -> RT_PHASE_END, finish() -> RT_MARCH_MISS
                if (PROF) prof[5]++;
                return 0;
            }
            reach = fmin(reach, pl.jump_limit);
        }
        const double mf = reach / pl.abs_step * (1.0 - 1e-9) - 2.0;
        if (mf >= (double)RT_MARCH_MIN_JUMP) return (long long)fmin(mf, 1.0e15);
        // inside the |g| < M zone or next to a range limit: plain steps, retry later
        if (PROF) prof[it > 0 ? 7 : 6]++;
        if (it > 0) {
            // A refinement level walks back over ONE step of the level before (<= ~100 steps of its own) towards a sign
            // change that is known to lie ahead, and |g| only shrinks on the way: a plan that stopped within a few
            // steps stopped at the band around that very crossing, and planning again before the crossing can only
            // find the same (it used to: 2.5 empty plans per hit ray on cornell_box, backing off 4, 8, 16 ... steps
            // through the last level, whose steps of 1e-8 are of the order of the band).  The sign change resets
            // cooldown (literal()).
            cooldown = 200;
            return 0;
        }
        cooldown = backoff;
        backoff = backoff * 2 < 64 ? backoff * 2 : 64;
        return 0;
    }
    __host__ __device__ __forceinline__ long long attempt_plan(Plan& pl) {
        plan_begin(pl);
        while (plan_hop(pl)) {
        }
        return plan_end(pl);
    }
    // nt / np: t and p after m more iterations (advance_exact of t by step and of p by sd)
    __host__ __device__ __forceinline__ void attempt_land(const Plan& pl, double nt, D3 np) {
        const double land = surface_func<KIND>(q, np);  // the reference's `r = next` at the landing sample
        n++;
        if (PROF) prof[2]++;
        const double x = (nt - t) - pl.shift;  // s[] is centred `shift` past the sample the jump started from
        double gp = pl.s[DEG];
#pragma unroll
        for (int k = DEG - 1; k >= 0; k--) gp = fma(gp, x, pl.s[k]);
        // self-check: the landing value must be what the polynomial predicts and keep the sign
        const bool same_sign = ((land > 0.0) == (r > 0.0)) && land != 0.0;
        if (same_sign && fabs(land - gp) <= 0.25 * pl.M && fabs(land) >= 0.5 * pl.M) {
            t = nt;
            p = np;
            r = land;
            backoff = 4;
            // A jump that ran up to the |g| = M boundary (or to the range limit) has nothing left to skip: the
            // next event is a few literal steps away.  Attempting again right away failed 4 times per ray
            // (half of all attempts, each a full plan); only a jump cut short by the span / hop limit retries.
            cooldown = pl.more ? 0 : RT_MARCH_LAND_COOLDOWN;
            return;
        }
        skip_ok = false;  // the model does not describe this ray: finish it with the plain loop
    }
    // the serial form (fused kernels, rt_intersect_batch)
    __host__ __device__ __forceinline__ void attempt() {
        Plan pl;
        const long long m = attempt_plan(pl);
        if (m <= 0) return;
        const double nt = advance_exact(t, step, m);
        D3 np;
        np.x = advance_exact(p.x, sd.x, m);
        np.y = advance_exact(p.y, sd.y, m);
        np.z = advance_exact(p.z, sd.z, m);
        attempt_land(pl, nt, np);
    }

    // the reference's literal step (ray_marching.rs:37-51)
    __host__ __device__ __forceinline__ void literal() {
        if (cooldown > 0) cooldown--;
        t += step;
        p.x += sd.x;
        p.y += sd.y;
        p.z += sd.z;
        const double next = surface_func<KIND>(q, p);
        n++;
        if (PROF) prof[it == 0 ? 0 : 1]++;
        if (approx_zero(next)) {
            it = depth;  // `finished`
            return;
        }
        if ((r < 0.0 && next > 0.0) || (r > 0.0 && next < 0.0)) {
            step *= -0.01;
            r = next;
            it++;
            sd = step * d;
            cooldown = 0;
            backoff = 4;
            return;
        }
        r = next;
    }
};

// `hull`: try the miss proof (3) when the ray starts.  The per-lane callers (k_intersect_batch, the fused k_bounce) pass
// false: a warp waits for its slowest lane there, which is a ray that hits, and the proof only adds to its work
// (cfg 2 on the cornell shape list: 509 -> 542 Mrays/s without it); the wavefront runs it in k_march_filter.
template <int KIND>
__host__ __device__ __forceinline__ bool march_loop_skip(const double* q, D3 o, D3 d, double start, double end, double min_t,
                                                         double max_t, double G, double F, double& t_out,
                                                         unsigned long long& evals, bool hull) {
    Marcher<KIND> m;
    m.begin(q, o, d, start, end, G, F, hull);
    int ph;
    while ((ph = m.phase()) != RT_PHASE_END) {
        if (ph == RT_PHASE_ATTEMPT) m.attempt();
        else m.literal();
    }
    evals += m.n;
    if (m.finish() == RT_MARCH_MISS) return false;
    if (m.t < min_t || m.t > max_t) return false;
    t_out = m.t;
    return true;
}

__host__ __device__ inline bool march_candidate_skip(const double* q, D3 o, D3 d, double start, double end, double min_t,
                                                     double max_t, double G, double F, double& t, unsigned long long& evals,
                                                     bool hull = false) {
    switch ((int)q[0]) {
        case RT_SURF_HEART: return march_loop_skip<RT_SURF_HEART>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
        case RT_SURF_SINE: return march_loop_skip<RT_SURF_SINE>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
        case RT_SURF_STAR: return march_loop_skip<RT_SURF_STAR>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
        case RT_SURF_DUPIN: return march_loop_skip<RT_SURF_DUPIN>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
        case RT_SURF_HUNTS: return march_loop_skip<RT_SURF_HUNTS>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
        default: return march_loop_skip<RT_SURF_CUSHION>(q, o, d, start, end, min_t, max_t, G, F, t, evals, hull);
    }
}

}  // namespace rt
