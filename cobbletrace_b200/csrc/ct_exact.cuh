// ct_exact.cuh -- device primitives that reproduce the reference's mixed fp64/fp32
// arithmetic bit for bit (SURVEY 0.2, 7 hard part #1).
//
// The reference computes vectors in double (v3_t, mymath.h:24-28), rounds every dot
// product / magnitude to float on return (mymath.h:229,213) and does its scalar work in
// float.  Every operation below is an explicit round-to-nearest intrinsic (__dmul_rn,
// __dadd_rn, __fmul_rn, ...): those are never contracted into FMAs, so the rounding points
// are the reference's whatever -fmad says.  B200 runs fp64 at half the fp32 rate, so exact
// evaluation is affordable; nothing here needs tensor cores.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace ct {

#define CT_DEV __device__ __forceinline__

constexpr float kRayTInit = 1e30f;              // ray_t.t of primary/shadow rays (raythread.cpp:508,304)
constexpr float kFinf = 4294967296.0f;          // FINF raythread.cpp:58
constexpr float kEps = 0.0001f;                 // bvh.cpp:152,161

struct V3 { double x, y, z; };

CT_DEV V3 vsub(V3 a, V3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }   // mymath.h:147
CT_DEV V3 vadd(V3 a, V3 b) { return {__dadd_rn(a.x, b.x), __dadd_rn(a.y, b.y), __dadd_rn(a.z, b.z)}; }   // mymath.h:129
CT_DEV V3 vscale(double s, V3 a) { return {__dmul_rn(s, a.x), __dmul_rn(s, a.y), __dmul_rn(s, a.z)}; }   // mymath.h:47
CT_DEV V3 vneg(V3 a) { return {-a.x, -a.y, -a.z}; }                                                      // mymath.h:118
CT_DEV V3 vcross(V3 a, V3 b) {                                                                           // mymath.h:234
    return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)),
            __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
            __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}
// DotProduct mymath.h:229: ((ax*bx + ay*by) + az*bz) in double, rounded to float on return.
CT_DEV float vdot(V3 a, V3 b) {
    return __double2float_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z)));
}
// Magnitude mymath.h:213: double sqrt, rounded to float on return.
CT_DEV float vmag(V3 a) {
    return __double2float_rn(__dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(a.x, a.x), __dmul_rn(a.y, a.y)), __dmul_rn(a.z, a.z))));
}

// mymath.h:11-17 macros: a NaN operand makes the comparison false and yields the SECOND operand.
CT_DEV float macro_min(float a, float b) { return (a < b) ? a : b; }
CT_DEV float macro_max(float a, float b) { return (a > b) ? a : b; }

// ---- rays ------------------------------------------------------------------------------------------
struct Ray {        // ray_t (scenefile.h:104-108)
    V3 o, d;
    float t;
};

// What the traversal loop keeps in registers: ray.t and the per-ray constants of the two certified fp32 filters
// (box_filter, tri_filter_miss).  The fp64 origin/direction the reference's own arithmetic needs stay in local
// memory (r64[0..2] = origin, r64[3..5] = direction, r64[6..8] = correctly rounded 1/direction once needed, r64[9] its
// state: < 0 not computed, 1 when some 1/d leaves the normal range) and are only touched when a filter cannot decide.
constexpr int kRay64 = 10;
struct TRay {
    float t;
    float rdf[3];   // float(1/d)
    float cl[3];    // round-down float of  -o/d - E   } E = per-axis bound on |filter quotient - reference quotient|,
    float cu[3];    // round-up   float of  -o/d + E   } see tray_setup
    float of[3], df[3];   // float(o), float(d)
    float cd;       // 2^-17 * max|d_i|, rounded up
    float om;       // max|o_i|, rounded up
    bool filt;      // false: some axis cannot be bounded (d == 0, non-finite, absurd magnitudes) -> exact slab tests only
    bool tfilt;     // false: magnitudes outside the range the triangle filter's error analysis covers
    float sg;       // tray_nearest_setup: the slop bound sigma of the order-free closest-hit search (k_primary_split), 0 = the ray may not take it
    double *r64;
};

// Per-ray setup of the filters.  bound[k] >= |b| for every node bound b on axis k (computed at upload;
// +inf when the tree holds non-finite or ill-ordered boxes, which disables the slab filter).
//
// For a node bound b on axis k the reference computes  q_ref = float( fl64( fl64(b - o) / d ) )   (bvh.cpp:166-175).
// With q* = (b - o)/d in real arithmetic, |q_ref - q*| <= (2^-24 + 2^-51) |q*|.
// The filter evaluates  y = bf * rdf + c  with  bf = float(b), rdf = float-reciprocal of float(d), c = fl64(-o * rdf):
//     rdf = (1/d)(1 + e),  |e| <= 2 * 2^-24 + 2^-47        (one rounding for float(d), one for the reciprocal)
//     |bf*rdf - b/d| <= 3.01 * 2^-24 |b/d| ,   |c - (-o/d)| <= 2.01 * 2^-24 |o/d|
// so |y - q_ref| <= 4.1 * 2^-24 * (|b| + |o|) / |d|  <=  E := 2^-21 * (bound + |o|) * |rdf| .
// cl / cu fold -E / +E into c, rounded DOWN / UP to float, and the filter's FMAs round down / up as well, so
//     fma_rd(bf, rdf, cl) <= q_ref <= fma_ru(bf, rdf, cu)          for every finite node bound.
// No fp64 division here: the correctly rounded 1/d that the division-free fp64 evaluation (box_times) wants is
// only computed when a ray first needs that path (ray64_reciprocals); r64[9] < 0 marks "not yet".
CT_DEV void tray_setup(TRay &r, const Ray &ray, const double bound[3], double *r64) {
    const double o[3] = {ray.o.x, ray.o.y, ray.o.z}, d[3] = {ray.d.x, ray.d.y, ray.d.z};
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const float df = __double2float_rn(d[k]);
        const float rdf = __frcp_rn(df);
        const double rd = (double)rdf;
        double c = __dmul_rn(-o[k], rd);
        double sum = __dadd_rn(bound[k], fabs(o[k]));
        double m = __dmul_rn(sum, fabs(rd));
        double e = __dmul_rn(m, 0x1p-21);
        // every quantity must be an ordinary number well inside the float range (a finite non-zero rdf rules out
        // d = 0, d = +-inf and directions outside the float range, NaNs fail the comparisons); magnitudes near the
        // float subnormals are left alone.  m < 2^99 also puts every quotient of a filtered ray below 1e30f
        // (pair_accept's T_FAR relies on it)
        ok = ok && (m < 0x1p99) && (fabs(rd) > 0x1p-100) && (fabs(rd) < 0x1p100) && (e > 0x1p-100) && (sum > 0x1p-60);
        r.rdf[k] = rdf;
        r.cl[k] = __double2float_rd(__dsub_rd(c, e));
        r.cu[k] = __double2float_ru(__dadd_ru(c, e));
        r.of[k] = __double2float_rn(o[k]);
        r.df[k] = df;
        r64[k] = o[k]; r64[3 + k] = d[k];
    }
    r64[9] = -1.0;
    r.filt = ok;
    double dm = fmax(fmax(fabs(d[0]), fabs(d[1])), fabs(d[2])), om = fmax(fmax(fabs(o[0]), fabs(o[1])), fabs(o[2]));
    r.tfilt = (dm >= 0x1p-20) && (dm <= 0x1p40) && (om <= 0x1p40);          // NaNs fail
    r.cd = __double2float_ru(__dmul_ru(dm, 0x1p-17));
    r.om = __double2float_ru(om);
    r.t = ray.t;
    r.sg = 0.0f;
    r.r64 = r64;
}

// Per-ray set-up of the ORDER-FREE closest-hit search (k_primary_split, ct_kernels.cuh): sigma, a bound on
//     tmin_ref(leaf box of Z) - t_ref(Z)
// over every triangle Z of the scene that passes the reference's barycentric test for this ray -- how much EARLIER than
// its own leaf's box a triangle can seem to be hit.  In real arithmetic that is <= 0 (a triangle lies inside the box of
// its leaf, UpdateNodeBounds bvh.cpp:30-49); what is left is rounding.  With eps = 2^-24, u = 2^-53, B = max bound[k]
// (>= every vertex coordinate), O = max|o_k|, D = max|d_k| and M = max_k (bound[k] + |o_k|) / |d_k| (>= every slab
// quotient of the ray and >= the t of any point inside the scene's box):
//   * IntersectTriangle (bvh.cpp:147-163) evaluates the determinants A, S, Q, T in fp64 from exact inputs -- six triple
//     products each, <= 6 roundings per term: |dA| <= 144 u D B^2, |dS|, |dQ| <= 72 u (O + B) D B, |dT| <= 144 u B^2 (O + B)
//     -- rounds each to float and multiplies by float(1 / a), |a| >= 1e-4 (1 - eps) (bvh.cpp:152).  Under the magnitude
//     limits below every |d.| / |A| <= 2^-20 (dT: relative to M), so the computed u, v, t are the true u*, v*, t* of the
//     plane intersection up to relative errors < 20 eps and absolute errors < 2^-20:
//         t_ref >= t* - 20 eps |t*| - 100 eps M ,   u* >= -17 eps, v* >= -17 eps, u* + v* <= 1 + 73 eps  (passes only);
//   * the point o + t* d = (1 - u* - v*) p1 + u* p2 + v* p3 therefore leaves the leaf's box by at most 107 eps times the
//     box's extent on any axis, i.e. t* >= (near quotient of axis k) - 107 eps * ext_k / |d_k| >= ... - 214 eps M;
//   * the reference's float tmin of the box exceeds the true entry distance by at most 1.01 eps M (tray_setup).
// Sum: < 340 eps M.  sigma = 512 eps M = 2^-15 M, rounded up; the slack also covers the float additions the walk does
// with it.  Rays outside the magnitude limits (or without a usable slab filter) get sigma = 0: they take the ordered walk.
CT_DEV void tray_nearest_setup(TRay &r, const double bound[3]) {
    r.sg = 0.0f;
    if (!r.filt) return;
    const double *o = r.r64, *d = r.r64 + 3;
    const double B = fmax(fmax(bound[0], bound[1]), bound[2]);
    const double O = fmax(fmax(fabs(o[0]), fabs(o[1])), fabs(o[2])), D = fmax(fmax(fabs(d[0]), fabs(d[1])), fabs(d[2]));
    double M = 0.0;
#pragma unroll
    for (int k = 0; k < 3; k++) M = fmax(M, (bound[k] + fabs(o[k])) * fabs((double)r.rdf[k]));      // rdf = (1/d)(1 + 2.01 eps)
    // 144 u D B^2 / 1e-4 <= 2^-20  <=>  D B^2 <= 2^12.7; the same for (O + B) D B; dT / |A| <= 100 eps M holds with M >= (B + O) / (2 D)
    const bool ok = (D * B * B <= 4096.0) && ((O + B) * D * B <= 4096.0) && (M > 0x1p-60) && (M < 0x1p60);
    if (ok) r.sg = __double2float_ru(M * (0x1p-15 * 1.000001));
}

// r64[6..8] = correctly rounded 1/d, r64[9] = 1 when some 1/d leaves the normal range (then box_times divides).
CT_DEV void ray64_reciprocals(double *r64) {
    bool odd = false;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const double d = r64[3 + k];
        r64[6 + k] = __ddiv_rn(1.0, d);
        // zero/inf/NaN directions are fine for the reciprocal form (IEEE gives the same inf/NaN quotients both ways);
        // only a finite non-zero d whose reciprocal leaves the normal range needs true divisions throughout
        const uint32_t hi = (uint32_t)__double2hiint(d), ex = (hi >> 20) & 0x7ffu;
        const bool zero = ((hi & 0x7fffffffu) | (uint32_t)__double2loint(d)) == 0u;
        odd = odd || (!zero && ex != 0x7ffu && (ex < 24u || ex > 2022u));
    }
    r64[9] = odd ? 1.0 : 0.0;
}

// ---- IntersectAABB (bvh.cpp:165-179) -------------------------------------------------------------------
// Literal arithmetic: six fp64 divisions, each rounded to float on assignment, macro min/max in float.
struct BoxTimes { float tmin, tmax; };
__device__ __noinline__ BoxTimes box_times_exact(double ox, double oy, double oz, double dx, double dy, double dz,
                                                 double nx, double ny, double nz, double mx, double my, double mz) {
    float tx1 = __double2float_rn(__ddiv_rn(__dsub_rn(nx, ox), dx));
    float tx2 = __double2float_rn(__ddiv_rn(__dsub_rn(mx, ox), dx));
    float tmin = macro_min(tx1, tx2);
    float tmax = macro_max(tx1, tx2);
    float ty1 = __double2float_rn(__ddiv_rn(__dsub_rn(ny, oy), dy));
    float ty2 = __double2float_rn(__ddiv_rn(__dsub_rn(my, oy), dy));
    tmin = macro_max(tmin, macro_min(ty1, ty2));
    tmax = macro_min(tmax, macro_max(ty1, ty2));
    float tz1 = __double2float_rn(__ddiv_rn(__dsub_rn(nz, oz), dz));
    float tz2 = __double2float_rn(__ddiv_rn(__dsub_rn(mz, oz), dz));
    tmin = macro_max(tmin, macro_min(tz1, tz2));
    tmax = macro_min(tmax, macro_max(tz1, tz2));
    return {tmin, tmax};
}

// mymath.h:11-17 on doubles (same NaN behaviour as the float macros).
CT_DEV double macro_min_d(double a, double b) { return (a < b) ? a : b; }
CT_DEV double macro_max_d(double a, double b) { return (a > b) ? a : b; }

// True when float(x) may differ from float(y) for some y within a few fp64 ulps of x: x sits within +-16 units of
// a float rounding boundary (the 29 dropped mantissa bits ~ 0x10000000), or x is non-zero with |x| < 2^-125 (float
// subnormal range, where the boundaries are elsewhere and the fp64 product may itself have lost bits).
CT_DEV bool float_rounding_unsafe(double x) {
    uint32_t lo = (uint32_t)__double2loint(x);
    uint32_t hi = (uint32_t)__double2hiint(x) & 0x7fffffffu;
    bool near_mid = ((lo & 0x1fffffffu) - 0x0ffffff0u) <= 0x20u;
    bool tiny = (hi < 0x38200000u) && ((hi | lo) != 0u);
    return near_mid | tiny;
}

// The two floats IntersectAABB compares, bit-exact (up to the sign of a zero, which no comparison sees), for ANY ray
// (r64 as laid out by tray_setup), usually without a division:
//   * rounding to float is monotonic and NaN-preserving, so taking the reference's macro min/max on the UNROUNDED
//     fp64 quotients and rounding only the two survivors gives the same float values (whenever the double
//     comparison picks a different operand than the float comparison would, both round to the same float);
//   * the quotient (b - o)/d is replaced by (b - o) * fl(1/d): each survivor is then within a few fp64 ulps of the
//     reference's double, so its float rounding can differ only if it lies that close to a float rounding boundary
//     (~2^-24 of tests) -- those, and rays whose 1/d leaves the normal range, redo the six true divisions.
CT_DEV BoxTimes box_times(double *r64, const double bmin[3], const double bmax[3]) {
    if (r64[9] < 0.0) ray64_reciprocals(r64);
    double x1 = __dmul_rn(__dsub_rn(bmin[0], r64[0]), r64[6]), x2 = __dmul_rn(__dsub_rn(bmax[0], r64[0]), r64[6]);
    double y1 = __dmul_rn(__dsub_rn(bmin[1], r64[1]), r64[7]), y2 = __dmul_rn(__dsub_rn(bmax[1], r64[1]), r64[7]);
    double z1 = __dmul_rn(__dsub_rn(bmin[2], r64[2]), r64[8]), z2 = __dmul_rn(__dsub_rn(bmax[2], r64[2]), r64[8]);
    double tmin = macro_min_d(x1, x2);
    double tmax = macro_max_d(x1, x2);
    tmin = macro_max_d(tmin, macro_min_d(y1, y2));
    tmax = macro_min_d(tmax, macro_max_d(y1, y2));
    tmin = macro_max_d(tmin, macro_min_d(z1, z2));
    tmax = macro_min_d(tmax, macro_max_d(z1, z2));
    if (float_rounding_unsafe(tmin) | float_rounding_unsafe(tmax) | (r64[9] != 0.0))
        return box_times_exact(r64[0], r64[1], r64[2], r64[3], r64[4], r64[5], bmin[0], bmin[1], bmin[2], bmax[0], bmax[1], bmax[2]);
    return {__double2float_rn(tmin), __double2float_rn(tmax)};
}

// The literal form, for callers that hold a plain Ray (KAT kernels).
CT_DEV BoxTimes box_times(const Ray &r, const double bmin[3], const double bmax[3]) {
    return box_times_exact(r.o.x, r.o.y, r.o.z, r.d.x, r.d.y, r.d.z, bmin[0], bmin[1], bmin[2], bmax[0], bmax[1], bmax[2]);
}

CT_DEV bool box_accept(BoxTimes b, float ray_t) { return b.tmax >= b.tmin && b.tmin < ray_t && b.tmax > 0.0f; }   // bvh.cpp:178

CT_DEV bool intersect_aabb(const Ray &r, const double bmin[3], const double bmax[3]) { return box_accept(box_times(r, bmin, bmax), r.t); }

// Certified fp32 filter for the slab test.  Brackets the reference's float tmin and tmax:
//     near_lo <= tmin_ref <= near_hi ,   far_lo <= tmax_ref <= far_hi
// (per axis the reference's min(t1,t2) is the quotient of the bound the ray meets first, because
// b -> q_ref(b) is monotone; max over axes of brackets brackets the max).  Only valid when r.filt.
struct BoxBracket { float near_lo, near_hi, far_lo, far_hi; };

CT_DEV BoxBracket box_filter(const TRay &r, const float bmin[3], const float bmax[3]) {
    float nl[3], nh[3], fl[3], fh[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const bool pos = r.rdf[k] > 0.0f;
        const float bn = pos ? bmin[k] : bmax[k], bf = pos ? bmax[k] : bmin[k];
        nl[k] = __fmaf_rd(bn, r.rdf[k], r.cl[k]);
        nh[k] = __fmaf_ru(bn, r.rdf[k], r.cu[k]);
        fl[k] = __fmaf_rd(bf, r.rdf[k], r.cl[k]);
        fh[k] = __fmaf_ru(bf, r.rdf[k], r.cu[k]);
    }
    BoxBracket b;
    b.near_lo = fmaxf(fmaxf(nl[0], nl[1]), nl[2]);
    b.near_hi = fmaxf(fmaxf(nh[0], nh[1]), nh[2]);
    b.far_lo = fminf(fminf(fl[0], fl[1]), fl[2]);
    b.far_hi = fminf(fminf(fh[0], fh[1]), fh[2]);
    return b;
}

// Verdicts that follow from the bracket alone (each is true only when certain; both false = undecided).
//   geometry:  tmax >= tmin && tmax > 0      (independent of ray.t)
//   distance:  tmin < ray.t
CT_DEV bool bracket_geom_yes(const BoxBracket &b) { return (b.far_lo >= b.near_hi) & (b.far_lo > 0.0f); }
CT_DEV bool bracket_geom_no(const BoxBracket &b) { return (b.far_hi < b.near_lo) | (b.far_hi <= 0.0f); }
CT_DEV bool bracket_t_yes(const BoxBracket &b, float ray_t) { return b.near_hi < ray_t; }
CT_DEV bool bracket_t_no(const BoxBracket &b, float ray_t) { return b.near_lo >= ray_t; }

// IntersectTriangle bvh.cpp:147-163 with edge1 = p2-p1, edge2 = p3-p1 precomputed at upload (the same
// two fp64 subtractions the reference redoes per call).  Returns the barycentric verdict; *t_out is
// the candidate distance (only meaningful when true).  The caller applies `if (t > 0.0001f) ray.t =
// min(ray.t, t)` -- the function returns true whatever the sign/size of t (SURVEY 0.4).
CT_DEV bool intersect_triangle(const Ray &r, V3 p1, V3 e1, V3 e2, float *t_out) {
    V3 h = vcross(r.d, e2);
    float a = vdot(e1, h);
    if (a > -kEps && a < kEps) return false;
    float f = __fdiv_rn(1.0f, a);
    V3 s = vsub(r.o, p1);
    float u = __fmul_rn(f, vdot(s, h));
    if (u < 0.0f || u > 1.0f) return false;
    V3 q = vcross(s, e1);
    float v = __fmul_rn(f, vdot(r.d, q));
    if (v < 0.0f || __fadd_rn(u, v) > 1.0f) return false;
    *t_out = __fmul_rn(f, vdot(e2, q));
    return true;
}

// Certified fp32 filter in front of IntersectTriangle (bvh.cpp:147-163).  Returns true only when the reference's
// test CERTAINLY has no effect on the traversal:
//   * it returns false (|a| < 1e-4, u outside [0,1], v < 0 or u + v > 1), or
//   * ANY_HIT only (shadow rays): it returns true but with t <= 1e-4, which never lowers ray.t (bvh.cpp:161) --
//     what a shadow ray leaving a surface sees of the triangle it starts on.
// Everything else (hits, near misses, out-of-range magnitudes) is left to the exact fp64 test.
//
// With A = e1.(d x e2), S = s.(d x e2), Q = d.(s x e1), T = e2.(s x e1), s = o - p1 in real arithmetic, the
// reference computes u = S/A, v = Q/A, t = T/A up to relative errors below 4.1 * 2^-24 (fp64 products, rounded to
// float, times float(1/a)).  Evaluating the same determinants in fp32 from float-rounded inputs gives
//     |A~ - A| <= EA = 2^-17 K1 K2 D        |S~ - S| <= ES = 2^-17 D K2 (O + K3)
//     |Q~ - Q| <= EQ = 2^-17 D K1 (O + K3)  |T~ - T| <= ET = 2^-17 K1 K2 (O + K3)
// with K1 = max|e1_i|, K2 = max|e2_i|, K3 = max|p1_i| (stored with the triangle, rounded up), D = max|d_i|,
// O = max|o_i| (worst case 67 * 2^-24 * magnitude each: input roundings, the float subtraction o - p1, five
// rounded operations per determinant).  A verdict is certified only with margins of twice these bounds, which
// also absorbs the reference's own float rounding of u, v, t (see DESIGN.md 2).  Magnitude limits (r.tfilt,
// finite K's in [2^-30, 2^30] -- else K1 is stored as NaN and nothing certifies) keep every product in the
// normal float range; ES, EQ >= 2^-40 keeps the reference's f * S from underflowing to -0.
// tri: 12 floats p1.xyz, K3, e1.xyz, K1, e2.xyz, K2.
template <bool ANY_HIT>
CT_DEV bool tri_filter_miss(const TRay &r, float4 t0, float4 t1, float4 t2) {
    const float k3 = t0.w, k1 = t1.w, k2 = t2.w;
    // h = d x e2, q = s x e1
    const float hx = __fmaf_rn(r.df[1], t2.z, -__fmul_rn(r.df[2], t2.y));
    const float hy = __fmaf_rn(r.df[2], t2.x, -__fmul_rn(r.df[0], t2.z));
    const float hz = __fmaf_rn(r.df[0], t2.y, -__fmul_rn(r.df[1], t2.x));
    const float sx = __fsub_rn(r.of[0], t0.x), sy = __fsub_rn(r.of[1], t0.y), sz = __fsub_rn(r.of[2], t0.z);
    const float A = __fmaf_rn(t1.x, hx, __fmaf_rn(t1.y, hy, __fmul_rn(t1.z, hz)));
    const float S = __fmaf_rn(sx, hx, __fmaf_rn(sy, hy, __fmul_rn(sz, hz)));
    const float qx = __fmaf_rn(sy, t1.z, -__fmul_rn(sz, t1.y));
    const float qy = __fmaf_rn(sz, t1.x, -__fmul_rn(sx, t1.z));
    const float qz = __fmaf_rn(sx, t1.y, -__fmul_rn(sy, t1.x));
    const float Q = __fmaf_rn(r.df[0], qx, __fmaf_rn(r.df[1], qy, __fmul_rn(r.df[2], qz)));
    const float sig = __fadd_ru(r.om, k3);                       // O + K3
    const float k12 = __fmul_ru(k1, k2);
    const float ea = __fmul_ru(k12, r.cd);
    const float es = fmaxf(__fmul_ru(__fmul_ru(r.cd, k2), sig), 0x1p-40f);
    const float eq = fmaxf(__fmul_ru(__fmul_ru(r.cd, k1), sig), 0x1p-40f);
    const float aa = fabsf(A);
    const bool tiny_a = __fadd_ru(aa, ea) < 9.9999e-05f;          // |a| < 1e-4 for certain (bvh.cpp:152)
    const bool sign_ok = aa > __fmul_ru(2.0f, ea);                // sign of a certain (false for NaN K1)
    const float Ss = A > 0.0f ? S : -S, Qs = A > 0.0f ? Q : -Q;   // oriented so that u = Ss/|A|, v = Qs/|A|
    bool miss = (Ss < -__fmul_ru(2.0f, es))                                                                        // u < 0
              | (Qs < -__fmul_ru(2.0f, eq))                                                                        // v < 0
              | (__fsub_rd(Ss, aa) > __fmul_ru(2.0f, __fadd_ru(es, ea)))                                           // u > 1
              | (__fsub_rd(__fadd_rd(Ss, Qs), aa) > __fmul_ru(2.0f, __fadd_ru(__fadd_ru(es, eq), ea)));            // u + v > 1
    if (ANY_HIT) {
        const float T = __fmaf_rn(t2.x, qx, __fmaf_rn(t2.y, qy, __fmul_rn(t2.z, qz)));
        const float Ts = A > 0.0f ? T : -T;
        const float et = __fmul_ru(__fmul_ru(k12, sig), 0x1p-16f);                    // 2 * ET
        // t <= 1e-4 for certain:  T <= 1e-4 (1 - 2^-20) |A|
        miss |= __fadd_ru(Ts, et) <= __fmul_rd(9.9999e-05f, __fsub_rd(aa, ea));
    }
    return tiny_a | (sign_ok & miss);
}

// ReflectRay raythread.cpp:270-273: 2.0*normal*Dot(normal,ray) - ray
CT_DEV V3 reflect_ray(V3 rv, V3 n) {
    double d = (double)vdot(n, rv);
    return vsub(vscale(d, vscale(2.0, n)), rv);
}

// pow(x, n) for ComputeLighting's specular term (raythread.cpp:321: pow(float, int) resolves to the double pow of glibc,
// whose result is the correctly rounded x^n except within ~2^-15 ulp of a rounding boundary -- its error bound is
// 0.52 ulp).  CUDA's pow() is documented at up to 2 ulp and does differ from glibc on reachable arguments (DESIGN 2), so
// for the integer exponents scene files hold (material_t.specular is an int) x^|n| is computed by square-and-multiply in
// double-double arithmetic, inverted in double-double for n < 0, and rounded once.  Each dd_mul / dd_recip is within
// 2^-104 relative, a squaring doubles the relative error it is given, so for |n| <= 2^31 the result is within 2^-72
// relative of x^n: the correctly rounded value unless x^n lies within 2^-19 ulp of a rounding boundary, and glibc's
// value wherever glibc is correctly rounded.  pow() is left to arguments that no float qv reaches with a finite result
// (x <= 2^-1000: 0, NaN) and to results outside [2^-900, 2^900] (an intermediate leaves that range), whose products
// with a float intensity never move the float accumulator.
struct DD { double hi, lo; };
CT_DEV DD dd_mul(DD a, DD b) {
    const double p = __dmul_rn(a.hi, b.hi);
    const double e = __fma_rn(a.hi, b.hi, -p);                                   // exact error of the product
    const double c = __dadd_rn(e, __dadd_rn(__dmul_rn(a.hi, b.lo), __dmul_rn(a.lo, b.hi)));
    const double hi = __dadd_rn(p, c);
    return {hi, __dadd_rn(__dsub_rn(p, hi), c)};                                 // fast two-sum: |p| >= |c|
}
// 1 / (a.hi + a.lo): q = fl(1/a.hi), then one Newton step with the exact remainder 1 - q a.hi
CT_DEV DD dd_recip(DD a) {
    const double q = __ddiv_rn(1.0, a.hi);
    const double rem = __fma_rn(-q, a.lo, __fma_rn(-q, a.hi, 1.0));
    const double c = __dmul_rn(rem, q);
    const double hi = __dadd_rn(q, c);
    return {hi, __dadd_rn(__dsub_rn(q, hi), c)};
}
CT_DEV double pow_int(double x, int n) {
    if (!(x > 0x1p-1000) || !(x < 0x1p1000)) return pow(x, (double)n);
    DD r = {1.0, 0.0}, b = {x, 0.0};
    for (uint32_t k = n < 0 ? 0u - (uint32_t)n : (uint32_t)n; k; k >>= 1) {
        if (k & 1u) r = dd_mul(r, b);
        if (k > 1u) b = dd_mul(b, b);
        if (!(fabs(b.hi) > 0x1p-900) || !(fabs(b.hi) < 0x1p900) || !(fabs(r.hi) > 0x1p-900) || !(fabs(r.hi) < 0x1p900))
            return pow(x, (double)n);                                            // leaves the range in which the error terms are normal numbers
    }
    if (n < 0) r = dd_recip(r);
    return __dadd_rn(r.hi, r.lo);
}

// raythread.cpp:321: intensity += li * pow(q, specular) -- the product in double, the sum rounded back to the float accumulator.
CT_DEV float specular_add(float intensity, float li, float q, int specular) {
    const double term = __dmul_rn((double)li, pow_int((double)q, specular));
    return __double2float_rn(__dadd_rn((double)intensity, term));
}

// ---- color.h ------------------------------------------------------------------------------------
CT_DEV uint32_t to_u8(float x) { return (uint32_t)__float2int_rz(x) & 0xffu; }   // float -> uint8_t argument conversion

// ColorToHsv (color.h:114) + `hsv.v = intensity` (raythread.cpp:365) + HsvToColor (color.h:122)
CT_DEV uint32_t shade_color(uint32_t color, float intensity) {
    float r = __fdiv_rn((float)(color & 0xffu), 255.0f);
    float g = __fdiv_rn((float)((color >> 8) & 0xffu), 255.0f);
    float b = __fdiv_rn((float)((color >> 16) & 0xffu), 255.0f);
    float max_c = macro_max(r, macro_max(g, b));
    float min_c = macro_min(r, macro_min(g, b));
    float delta = __fsub_rn(max_c, min_c);
    float s, h;
    if (max_c != 0.0f) {
        s = __fdiv_rn(delta, max_c);
        if (r == max_c) h = __fdiv_rn(__fsub_rn(g, b), delta);
        else if (g == max_c) h = __fadd_rn(2.0f, __fdiv_rn(__fsub_rn(b, r), delta));
        else h = __fadd_rn(4.0f, __fdiv_rn(__fsub_rn(r, g), delta));
        h = __double2float_rn(__dmul_rn((double)h, 60.0));
        if (h < 0.0f) h = __double2float_rn(__dadd_rn((double)h, 360.0));
    } else {
        s = 0.0f; h = -1.0f;
    }
    float v = intensity;
    float R, G, B;
    if (s == 0.0f) {
        R = G = B = v;
    } else {
        h = __double2float_rn(__ddiv_rn((double)h, 60.0));
        int i = (int)floor((double)h);
        float f = __fsub_rn(h, (float)i);
        float aa = __fmul_rn(v, __fsub_rn(1.0f, s));
        float bb = __fmul_rn(v, __fsub_rn(1.0f, __fmul_rn(s, f)));
        float cc = __fmul_rn(v, __fsub_rn(1.0f, __fmul_rn(s, __fsub_rn(1.0f, f))));
        R = G = B = 0.0f;
        switch (i) {
        case 0: R = v;  G = cc; B = aa; break;
        case 1: R = bb; G = v;  B = aa; break;
        case 2: R = aa; G = v;  B = cc; break;
        case 3: R = aa; G = bb; B = v;  break;
        case 4: R = cc; G = aa; B = v;  break;
        case 5: R = v;  G = aa; B = bb; break;
        }
    }
    uint32_t r8 = to_u8(macro_min(__fmul_rn(R, 255.0f), 255.0f));
    uint32_t g8 = to_u8(macro_min(__fmul_rn(G, 255.0f), 255.0f));
    uint32_t b8 = to_u8(macro_min(__fmul_rn(B, 255.0f), 255.0f));
    return (b8 << 16) | (g8 << 8) | r8;
}

// The low byte of the reference's (int)c on x86-64: cvttsd2si truncates toward zero and returns the "integer indefinite" value
// 0x80000000 (low byte 0) for a NaN and for every c outside (-2^31 - 1, 2^31).  PTX's cvt.rzi.s32.f64 saturates instead
// (c >= 2^31 gives 0x7fffffff, low byte 0xff), so those values are mapped here.
CT_DEV uint32_t x86_double_to_int_low8(double c) {
    return (c > -2147483649.0 && c < 2147483648.0) ? ((uint32_t)__double2int_rz(c) & 0xffu) : 0u;
}

// raythread.cpp:375-379: local*(1-r) + reflected*r per channel in double, truncated to uint8_t
CT_DEV uint32_t blend_color(uint32_t lc, uint32_t rc, float reflection) {
    double wl = (double)__fsub_rn(1.0f, reflection), wr = (double)reflection;
    uint32_t out = 0;
#pragma unroll
    for (int sh = 0; sh <= 16; sh += 8) {
        double l = (double)((lc >> sh) & 0xffu), r = (double)((rc >> sh) & 0xffu);
        double c = __dadd_rn(__dmul_rn(wl, l), __dmul_rn(wr, r));
        out |= x86_double_to_int_low8(c) << sh;
    }
    return out;
}

}  // namespace ct
