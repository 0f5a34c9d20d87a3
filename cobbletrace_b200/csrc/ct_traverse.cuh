// ct_traverse.cuh -- record loads, the exact (fp64) fallbacks behind the certified filters, and the three BVH walks
// (traverse_closest: IntersectBVHClosest in the reference's visit order; traverse_early: any-hit and first-line walks with deferred leaves).
// Part of the single translation unit ct_gpu.cu (everything lives in its anonymous namespace).
#pragma once

#include "ct_layout.cuh"

namespace {

CT_DEV V3 ld3(const double *p) { return {p[0], p[1], p[2]}; }

CT_DEV void load_tri(const DevTri *tris, uint32_t pos, V3 &p1, V3 &e1, V3 &e2) {
    const double2 *p = reinterpret_cast<const double2 *>(tris + pos);
    double2 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3);
    double e = __ldg(reinterpret_cast<const double *>(p + 4));
    p1 = {a.x, a.y, b.x};
    e1 = {b.y, c.x, c.y};
    e2 = {d.x, d.y, e};
}

// Optional (CT_PREFETCH=1): request the records of a pair's children as soon as the pair has arrived, so that their
// latency overlaps this visit's slab tests.  Measured neutral-to-negative on full frames (the walks are issue
// bound there), kept as a build-time experiment.
CT_DEV void prefetch_children(const Params &P, const DevPair32 &pr) {
#if defined(CT_PREFETCH) && CT_PREFETCH
    const char *l = pr.l_cnt ? reinterpret_cast<const char *>(P.tris32 + pr.l_ref) : reinterpret_cast<const char *>(P.pairs32 + pr.l_ref);
    const char *r = pr.r_cnt ? reinterpret_cast<const char *>(P.tris32 + pr.r_ref) : reinterpret_cast<const char *>(P.pairs32 + pr.r_ref);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(l)); asm volatile("prefetch.global.L2 [%0];" ::"l"(l + 32));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(r)); asm volatile("prefetch.global.L2 [%0];" ::"l"(r + 32));
#endif
}

// 32 bytes per lane in ONE load instruction (ld.global.nc.v8 -> LDG.E.256, new with sm_100): a whole child of a wide
// node, half a child pair.  The lanes of a walking warp read 32 different records, so every load instruction costs the
// L1 one tag look-up per lane whatever its width -- the walks are bound by exactly that (l1tex throughput 79 % of peak in
// k_shadow) -- and a 256-bit load halves the look-ups per record.  -DCT_LDG256=0: two 128-bit loads.  p: 32-byte aligned.
#ifndef CT_LDG256
#define CT_LDG256 1
#endif
CT_DEV void ldg256(const void *p, float4 &a, uint4 &b) {
#if CT_LDG256
    uint32_t x0, x1, x2, x3;
    asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(x0), "=r"(x1), "=r"(x2), "=r"(x3), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
    a = make_float4(__uint_as_float(x0), __uint_as_float(x1), __uint_as_float(x2), __uint_as_float(x3));
#else
    a = __ldg(reinterpret_cast<const float4 *>(p));
    b = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
#endif
}

CT_DEV void load_pair32(const DevPair32 *pairs, uint32_t pid, DevPair32 &p) {
    float4 a, c; uint4 bu, m;
    ldg256(pairs + pid, a, bu);
    ldg256(reinterpret_cast<const char *>(pairs + pid) + 32, c, m);
    const float4 b = make_float4(__uint_as_float(bu.x), __uint_as_float(bu.y), __uint_as_float(bu.z), __uint_as_float(bu.w));
    p.lmin[0] = a.x; p.lmin[1] = a.y; p.lmin[2] = a.z; p.lmax[0] = a.w; p.lmax[1] = b.x; p.lmax[2] = b.y;
    p.rmin[0] = b.z; p.rmin[1] = b.w; p.rmin[2] = c.x; p.rmax[0] = c.y; p.rmax[1] = c.z; p.rmax[2] = c.w;
    p.l_ref = m.x; p.l_cnt = m.y; p.r_ref = m.z; p.r_cnt = m.w;
}

// ---- cold paths: the reference's own fp64 arithmetic, out of line so that its operands only occupy registers
// while it runs.  `r64` = the ray's origin (0..2) and direction (3..5) in local memory.
__device__ __noinline__ BoxTimes exact_child(const DevPair64 *pairs, uint32_t pid, uint32_t side, double *r64) {
    const double2 *q = reinterpret_cast<const double2 *>(pairs + pid) + 3u * side;
    double2 a = __ldg(q), b = __ldg(q + 1), c = __ldg(q + 2);
    const double bmin[3] = {a.x, a.y, b.x}, bmax[3] = {b.y, c.x, c.y};
    return box_times(r64, bmin, bmax);
}

CT_DEV bool exact_root(const Params &P, double *r64, float ray_t) {
    return box_accept(box_times(r64, P.root_min, P.root_max), ray_t);
}

// IntersectAABB's verdict for the root box: the fp32 bracket when it is certain, the fp64 arithmetic otherwise.
CT_DEV bool root_accept(const Params &P, const TRay &r) {
    if (r.filt) {
        const BoxBracket b = box_filter(r, P.root_min32, P.root_max32);
        if (bracket_geom_no(b) | bracket_t_no(b, r.t)) return false;
        if (bracket_geom_yes(b) & bracket_t_yes(b, r.t)) return true;
    }
    return exact_root(P, r.r64, r.t);
}

struct TriHit { bool hit; float t; };
__device__ __noinline__ TriHit tri_exact(const DevTri *tris, uint32_t pos, const double *r64) {
    V3 p1, e1, e2;
    load_tri(tris, pos, p1, e1, e2);
    Ray r;
    r.o = {r64[0], r64[1], r64[2]}; r.d = {r64[3], r64[4], r64[5]}; r.t = 0.0f;
    TriHit h;
    h.t = 0.0f;
    h.hit = intersect_triangle(r, p1, e1, e2, &h.t);
    return h;
}

// IntersectTriangle's verdict for the triangle at `pos`: the fp32 filter discards what certainly has no effect,
// the fp64 arithmetic decides the rest.
template <bool ANY_HIT, bool COUNT>
CT_DEV TriHit leaf_triangle(const Params &P, const TRay &r, uint32_t pos, LocalCount &lc) {
    const float4 *q = reinterpret_cast<const float4 *>(P.tris32 + pos);
    const bool miss = tri_filter_miss<ANY_HIT>(r, __ldg(q), __ldg(q + 1), __ldg(q + 2));
    if (r.tfilt & miss) return {false, 0.0f};
    if (COUNT) lc.tri_exact++;
    return tri_exact(P.tris, pos, r.r64);
}

// IntersectAABB's verdicts for the two children of pair `pid`, bit-exact: the fp32 brackets decide when they
// can (no branch on the way), the fp64 arithmetic otherwise.  On return [r_lo, r_hi] brackets the reference's
// tmin of the RIGHT child (collapsed to the exact value when the fp64 path ran), which is what its deferred
// `tmin < ray.t` re-check needs.
// T_FAR: the caller's ray.t is 1e30f for good (shadow rays); a filtered ray has |quotients| < 2^99 < 1e30 (tray_setup),
// so `tmin < ray.t` needs no test.
template <bool COUNT, bool T_FAR = false>
CT_DEV void pair_accept(const Params &P, const TRay &r, uint32_t pid, const DevPair32 &pr, bool &hit_l, bool &hit_r,
                        float &r_lo, float &r_hi, LocalCount &lc) {
    const BoxBracket bl = box_filter(r, pr.lmin, pr.lmax), br = box_filter(r, pr.rmin, pr.rmax);
    const bool no_l = T_FAR ? bracket_geom_no(bl) : (bracket_geom_no(bl) | bracket_t_no(bl, r.t));
    const bool yes_l = T_FAR ? bracket_geom_yes(bl) : (bracket_geom_yes(bl) & bracket_t_yes(bl, r.t));
    const bool no_r = T_FAR ? bracket_geom_no(br) : (bracket_geom_no(br) | bracket_t_no(br, r.t));
    const bool yes_r = T_FAR ? bracket_geom_yes(br) : (bracket_geom_yes(br) & bracket_t_yes(br, r.t));
    hit_l = yes_l; hit_r = yes_r;
    r_lo = br.near_lo; r_hi = br.near_hi;
    const bool open_l = !r.filt | !(no_l | yes_l), open_r = !r.filt | !(no_r | yes_r);
    if (open_l | open_r) {
        if (open_l) {
            if (COUNT) lc.box_exact++;
            hit_l = box_accept(exact_child(P.pairs64, pid, 0u, r.r64), r.t);
        }
        if (open_r) {
            if (COUNT) lc.box_exact++;
            BoxTimes e = exact_child(P.pairs64, pid, 1u, r.r64);
            r_lo = r_hi = e.tmin;
            hit_r = box_accept(e, r.t);
        }
    }
}

// The early-exit walks on a NESTED tree (every child's box inside its parent's box, bit for bit -- what UpdateNodeBounds,
// bvh.cpp:30-49, produces: a node's box is the min / max over its own triangles' vertices, and a child's triangles are a
// subset of its parent's; checked at upload) only need a CONSERVATIVE box test.  With ray.t fixed (1e30f or 0 until the
// walk ends) and no NaN among the slab quotients (r.filt: no zero direction component), the reference's floats are
// monotone in the box:  q(b) = float(fl64(fl64(b - o) / d))  is a monotone function of the bound b, so per axis the
// parent's near quotient <= the child's and its far quotient >= the child's, hence
//     tmin(parent) <= tmin(child)   and   tmax(parent) >= tmax(child)
// and IntersectAABB's verdict (tmax >= tmin && tmin < ray.t && tmax > 0, bvh.cpp:178) for a child implies the same verdict
// for its parent, grand-parent, ... up to the root.  "The reference's walk reaches this leaf" is therefore equivalent to
// "the leaf's OWN box passes IntersectAABB", whatever happened on the way down.  So the walk may accept any superset of
// the boxes the reference accepts -- it only has to find the candidate leaves; a triangle that passes the exact test
// counts if its leaf's box passes the exact slab test (candidate_reached, one fp64 box test per candidate instead of
// exact verdicts for every box of the walk).  pair_maybe is that superset test: the lower end of the near bracket and
// the upper end of the far bracket of box_filter, i.e. half its FMAs, no undecided case, no fp64 fallback, no branch.
template <bool T_FAR>
CT_DEV bool box_maybe(const TRay &r, const float bmin[3], const float bmax[3]) {
    float nl[3], fh[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const bool pos = r.rdf[k] > 0.0f;
        nl[k] = __fmaf_rd(pos ? bmin[k] : bmax[k], r.rdf[k], r.cl[k]);       // <= the reference's near quotient on this axis
        fh[k] = __fmaf_ru(pos ? bmax[k] : bmin[k], r.rdf[k], r.cu[k]);       // >= its far quotient
    }
    const float near_lo = fmaxf(fmaxf(nl[0], nl[1]), nl[2]), far_hi = fminf(fminf(fh[0], fh[1]), fh[2]);
    const bool no = T_FAR ? ((far_hi < near_lo) | (far_hi <= 0.0f)) : ((far_hi < near_lo) | (far_hi <= 0.0f) | (near_lo >= r.t));
    return !no;                                                              // false only when the reference certainly rejects
}

// Does the reference's walk reach the leaf that holds the triangle at `pos`?  (nested tree, r.filt: see above)
CT_DEV bool candidate_reached(const Params &P, const TRay &r, uint32_t pos) {
    const uint32_t code = __ldg(P.tri_parent + pos);                         // 2 * pair + side of the leaf's box
    if (code == kNoPos) return exact_root(P, r.r64, r.t);                    // the root itself is the leaf
    return box_accept(exact_child(P.pairs64, code >> 1, code & 1u, r.r64), r.t);
}

enum TraverseMode { kClosest, kAnyHit, kFirstLine };
enum { kTravMiss = 0, kTravHit = 1, kTravOverBudget = -1 };

constexpr uint32_t kFullMask = 0xffffffffu;

// Build-time bounds checks (-DCT_DEBUG_BOUNDS=1; compute-sanitizer is not available on every pool): trap with a message.
#if defined(CT_DEBUG_BOUNDS) && CT_DEBUG_BOUNDS
#define CT_CHECK(cond) do { if (!(cond)) { printf("CT_CHECK failed: %s (line %d)\n", #cond, __LINE__); __trap(); } } while (0)
#else
#define CT_CHECK(cond) do { } while (0)
#endif

// IntersectBVHClosest (bvh.cpp:198-222) as an explicit-stack DFS in the reference's visit order (left subtree,
// then right) -- the closest-hit walk of primary rays and of ct_gpu_debug_closest (any initial ray.t).
// The reference tests a node's box when it VISITS the node; here both children of a passing interior node are
// fetched and tested together (one 64-byte fetch, two independent slab tests in flight):
//   * the left child is visited next, so "now" is its visit time;
//   * the right child's tmin/tmax do not depend on ray.t; of the three accept conditions (bvh.cpp:178) only
//     `tmin < ray.t` does, and ray.t only ever decreases -- so a right child failing now fails at visit time too
//     and is dropped, and one that passes now is pushed WITH (a bracket of) its tmin and re-checked against the
//     then-current ray.t when popped.  Same boxes accepted, same triangles tested in the same order, same counts.
// Leaves are tested on the spot: ray.t must be up to date for the next box (an early-exit walk may defer them,
// traverse_early; this one may not, and for the same reason it cannot be parked and finished out of order).
// WARP-SYNCHRONOUS: all 32 lanes call it (lanes without a ray pass active = false); every iteration = one node
// visit per live lane, and the lanes re-converge at the vote that ends it (left to itself the compiler lets the
// lanes of a warp drift apart for the whole walk: measured 8 of 32 lanes active).
// Returns kTravHit/kTravMiss = ray.t != 1e30f ("found"), or kTravOverBudget when the walk was given up after `budget` pair visits
// (k_primary then parks the ray for k_primary_long: warps made of long walks only).
#ifndef CT_SM_CLOSEST
#define CT_SM_CLOSEST 0
#endif
constexpr int kSmClosest = CT_SM_CLOSEST;                         // stack entries of the closest-hit walk kept in shared memory
constexpr int kClosestWords = kSmClosest > 0 ? 5 * kSmClosest : 1;   // k_primary declares closest_sm[kClosestWords * kBlockThreads]
#ifndef CT_LEAF_HOLD
#define CT_LEAF_HOLD 0
#endif
constexpr int kLeafHold = CT_LEAF_HOLD;
template <bool COUNT, bool BUDGETED = false>
CT_DEV int traverse_closest(const Params &P, TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc, uint32_t *sm = nullptr,
                            const uint32_t budget = 0xffffffffu) {
    // stack entry = a pushed right child: (ref, cnt), the bracket of its tmin and its parent pair (to find its fp64
    // bounds again when the bracket cannot decide).  The first kSmClosest entries live in shared memory (sm = this thread's
    // column of the kernel's closest_sm array, five words per entry; see traverse_wide for the why), the rest in local memory.
    constexpr int kSm = kSmClosest;
    uint32_t stk_ref[kStackMax - kSm], stk_cnt[kStackMax - kSm], stk_src[kStackMax - kSm];
    float stk_lo[kStackMax - kSm], stk_hi[kStackMax - kSm];
    auto sm_at = [&](int i, int w) -> uint32_t & { return sm[(5 * i + w) * kBlockThreads]; };
    int sp = 0;
    uint32_t visits = 0;       // pair visits so far
    bool over = false;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;      // "closestIndex = 0" default, resolved by the caller via pos_of_tri0
    uint32_t cur_ref = P.root_ref, cur_cnt = P.root_cnt;   // current (already accepted) node
    bool live = false;
    if (active) {
        if (COUNT) lc.box++;
        live = root_accept(P, r);
    }
    while (__any_sync(kFullMask, live)) {
        // -DCT_LEAF_HOLD=K (experiment): a lane that has reached a leaf waits until K lanes hold one (or nobody is left to
        // walk), so that the triangle tests -- which otherwise run in most iterations for a handful of lanes -- are shared
        bool hold = false;
        if (kLeafHold > 0) {
            const uint32_t at_leaf = __ballot_sync(kFullMask, live & (cur_cnt > 0)), walking = __ballot_sync(kFullMask, live & (cur_cnt == 0));
            hold = walking != 0u && __popc(at_leaf) < kLeafHold;
        }
        if (live) {
            bool need_pop = true;
            if (cur_cnt > 0) {
                if (hold) need_pop = false;
                else for (uint32_t i = 0; i < cur_cnt; i++) {
                    uint32_t pos = cur_ref + i;
                    if (COUNT) lc.tri++;
                    const TriHit th = leaf_triangle<false, COUNT>(P, r, pos, lc);
                    if (th.hit) {
                        if (th.t > kEps) r.t = macro_min(r.t, th.t);               // bvh.cpp:161
                        if (r.t != kRayTInit && r.t < tclosest) {                  // bvh.cpp:212
                            closest_pos = pos; tclosest = r.t;
                        }
                    }
                }
            } else {
                CT_CHECK(cur_ref < P.n_pairs);
                if (BUDGETED && ++visits > budget) { over = true; live = false; continue; }      // a long walk: the caller parks the ray (k_primary<COUNT, true>)
                DevPair32 pr;
                load_pair32(P.pairs32, cur_ref, pr);
                prefetch_children(P, pr);
                if (COUNT) lc.box += 2;
                bool hit_l, hit_r; float r_lo, r_hi;
                pair_accept<COUNT>(P, r, cur_ref, pr, hit_l, hit_r, r_lo, r_hi, lc);
                if (hit_l & hit_r) {
                    CT_CHECK(sp < kStackMax);
                    if (sp < kSm) {
                        sm_at(sp, 0) = pr.r_ref; sm_at(sp, 1) = pr.r_cnt; sm_at(sp, 2) = cur_ref;
                        sm_at(sp, 3) = __float_as_uint(r_lo); sm_at(sp, 4) = __float_as_uint(r_hi);
                    } else {
                        const int k = sp - kSm;
                        stk_ref[k] = pr.r_ref; stk_cnt[k] = pr.r_cnt; stk_lo[k] = r_lo; stk_hi[k] = r_hi; stk_src[k] = cur_ref;
                    }
                    sp++;
                }
                if (hit_l | hit_r) {
                    cur_ref = hit_l ? pr.l_ref : pr.r_ref; cur_cnt = hit_l ? pr.l_cnt : pr.r_cnt;
                    need_pop = false;
                }
            }
            if (need_pop) {
                live = false;
                while (sp > 0) {
                    --sp;
                    const bool in_sm = sp < kSm;
                    const int k = sp - kSm;
                    const float lo = in_sm ? __uint_as_float(sm_at(sp, 3)) : stk_lo[k];
                    if (lo >= r.t) continue;                                  // the deferred `tmin < ray.t` of bvh.cpp:178
                    const float hi = in_sm ? __uint_as_float(sm_at(sp, 4)) : stk_hi[k];
                    if (!(hi < r.t)) {
                        if (COUNT) lc.box_exact++;
                        BoxTimes e = exact_child(P.pairs64, in_sm ? sm_at(sp, 2) : stk_src[k], 1u, r.r64);
                        if (!(e.tmin < r.t)) continue;
                    }
                    cur_ref = in_sm ? sm_at(sp, 0) : stk_ref[k]; cur_cnt = in_sm ? sm_at(sp, 1) : stk_cnt[k]; live = true;
                    break;
                }
            }
        }
    }
    if (!active) return kTravMiss;
    if (BUDGETED && over) return kTravOverBudget;          // given up after `budget` pair visits: ray.t, tclosest, closest_pos are those of a walk half done
    return r.t != kRayTInit ? kTravHit : kTravMiss;
}

// The same walk with CONSERVATIVE tests at the interior boxes (nested tree, r.filt: see box_maybe above).  The reference
// reaches a leaf iff the leaf's OWN box passes IntersectAABB against the ray.t of that moment, whatever happened on the way
// down -- so the boxes on the way only have to be accepted whenever the reference accepts them (box_maybe: the lower end of
// the near bracket, the upper end of the far bracket: half the FMAs of pair_accept, no undecided case, no fp64 fallback),
// and the exact verdict (certified bracket, fp64 when it cannot decide) is needed once per leaf the walk OPENS, against
// the ray.t of that moment, from the leaf's own bounds in its parent's pair record.  The visit order stays the reference's
// (left subtree first; a right child is pushed with the lower end of its near bracket and dropped when popped if ray.t
// has fallen to it), so the leaves are scanned in DFS order with the reference's ray.t: same triangles tested in the same
// order, same ray.t / tclosest / closestIndex.  Box-test COUNTS are this walk's own (a superset of the reference's boxes).
// WARP-SYNCHRONOUS; lanes whose ray does not allow conservative tests pass active = false and take traverse_closest.
template <bool T_FAR>
CT_DEV bool box_maybe_lo(const TRay &r, const float bmin[3], const float bmax[3], float &near_lo) {
    float nl[3], fh[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const bool pos = r.rdf[k] > 0.0f;
        nl[k] = __fmaf_rd(pos ? bmin[k] : bmax[k], r.rdf[k], r.cl[k]);
        fh[k] = __fmaf_ru(pos ? bmax[k] : bmin[k], r.rdf[k], r.cu[k]);
    }
    near_lo = fmaxf(fmaxf(nl[0], nl[1]), nl[2]);
    const float far_hi = fminf(fminf(fh[0], fh[1]), fh[2]);
    const bool no = T_FAR ? ((far_hi < near_lo) | (far_hi <= 0.0f)) : ((far_hi < near_lo) | (far_hi <= 0.0f) | (near_lo >= r.t));
    return !no;
}

template <bool COUNT>
CT_DEV int traverse_closest_cons(const Params &P, TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc) {
    uint32_t stk_ref[kStackMax], stk_cnt[kStackMax], stk_src[kStackMax];      // a pushed right child: (ref, cnt), its parent pair
    float stk_lo[kStackMax];                                                  // ... and the lower end of its near bracket
    int sp = 0;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;
    uint32_t cur_ref = P.root_ref, cur_cnt = P.root_cnt, cur_code = kNoPos;   // code = 2 * pair + side of the node's own box (kNoPos: the root)
    bool live = false;
    if (active) {
        if (COUNT) lc.box++;
        live = root_accept(P, r);
    }
    while (__any_sync(kFullMask, live)) {
        if (live) {
            bool need_pop = true;
            if (cur_cnt > 0) {
                bool acc = true;                                              // (the root itself: accepted above)
                if (cur_code != kNoPos) {                                     // IntersectAABB for the leaf's own box, now
                    const uint32_t pid = cur_code >> 1, side = cur_code & 1u;
                    const float4 *q = reinterpret_cast<const float4 *>(P.pairs32 + pid);
                    const float4 x = __ldg(q + side), y = __ldg(q + 1 + side);      // left: floats 0..5, right: floats 6..11
                    float bmin[3], bmax[3];
                    if (side == 0u) { bmin[0] = x.x; bmin[1] = x.y; bmin[2] = x.z; bmax[0] = x.w; bmax[1] = y.x; bmax[2] = y.y; }
                    else { bmin[0] = x.z; bmin[1] = x.w; bmin[2] = y.x; bmax[0] = y.y; bmax[1] = y.z; bmax[2] = y.w; }
                    const BoxBracket bb = box_filter(r, bmin, bmax);
                    const bool no = bracket_geom_no(bb) | bracket_t_no(bb, r.t), yes = bracket_geom_yes(bb) & bracket_t_yes(bb, r.t);
                    acc = yes;
                    if (!(no | yes)) {
                        if (COUNT) lc.box_exact++;
                        acc = box_accept(exact_child(P.pairs64, pid, side, r.r64), r.t);
                    }
                }
                if (acc) {
                    for (uint32_t i = 0; i < cur_cnt; i++) {
                        uint32_t pos = cur_ref + i;
                        if (COUNT) lc.tri++;
                        const TriHit th = leaf_triangle<false, COUNT>(P, r, pos, lc);
                        if (th.hit) {
                            if (th.t > kEps) r.t = macro_min(r.t, th.t);               // bvh.cpp:161
                            if (r.t != kRayTInit && r.t < tclosest) {                  // bvh.cpp:212
                                closest_pos = pos; tclosest = r.t;
                            }
                        }
                    }
                }
            } else {
                CT_CHECK(cur_ref < P.n_pairs);
                DevPair32 pr;
                load_pair32(P.pairs32, cur_ref, pr);
                if (COUNT) lc.box += 2;
                float l_lo, r_lo;
                const bool hit_l = box_maybe_lo<false>(r, pr.lmin, pr.lmax, l_lo), hit_r = box_maybe_lo<false>(r, pr.rmin, pr.rmax, r_lo);
                if (hit_l & hit_r) {
                    CT_CHECK(sp < kStackMax);
                    stk_ref[sp] = pr.r_ref; stk_cnt[sp] = pr.r_cnt; stk_lo[sp] = r_lo; stk_src[sp] = cur_ref;
                    sp++;
                }
                if (hit_l | hit_r) {
                    cur_code = 2u * cur_ref + (hit_l ? 0u : 1u);
                    cur_ref = hit_l ? pr.l_ref : pr.r_ref; cur_cnt = hit_l ? pr.l_cnt : pr.r_cnt;
                    need_pop = false;
                }
            }
            if (need_pop) {
                live = false;
                while (sp > 0) {
                    --sp;
                    if (stk_lo[sp] >= r.t) continue;                          // tmin >= its lower bracket end >= ray.t: bvh.cpp:178 rejects it now
                    cur_ref = stk_ref[sp]; cur_cnt = stk_cnt[sp]; cur_code = 2u * stk_src[sp] + 1u; live = true;
                    break;
                }
            }
        }
    }
    if (!active) return kTravMiss;
    return r.t != kRayTInit ? kTravHit : kTravMiss;
}

// The same walk with LANE REFILL (north_star: "__ballot_sync / __shfl_sync compaction for ray regrouping"): the warp
// does not wait for the slowest ray of a group of 32.  A lane whose walk has ended hands its result to the job and falls
// idle; as soon as kRefillLanes lanes are idle (one ballot per iteration) the job deals new rays to exactly those lanes --
// ranked with a prefix popcount over the idle mask -- whose set-up then runs for that many lanes at once.  Per ray nothing
// changes (same visits, same order, same arithmetic); what changes is which rays share a warp at any moment.  Besides the
// fuller warps this removes the per-group barrier, so a kernel ends with its longest single WALK, not its slowest group.
// A JOB supplies the rays and takes the results:
//     bool refill(P, idle_mask, got, r, r64)   warp-uniform.  May hand a ray to any lane of idle_mask: sets got and fills
//                                              r / r64 (tray_setup).  Returns false once the source is exhausted.
//     void finish(P, found, tc, pos)           per lane, when its walk has ended.
#ifndef CT_REFILL_T
#define CT_REFILL_T 0                 // 0: off (k_primary walks whole chunks); 1..32: idle lanes that trigger a refill
#endif
constexpr int kRefillLanes = CT_REFILL_T > 0 ? CT_REFILL_T : 32;
template <bool COUNT, class Job>
CT_DEV void traverse_closest_refill(const Params &P, Job &job, LocalCount &lc) {
    uint32_t stk_ref[kStackMax], stk_cnt[kStackMax], stk_src[kStackMax];
    float stk_lo[kStackMax], stk_hi[kStackMax];
    int sp = 0;
    float tclosest = kFinf;
    uint32_t closest_pos = kNoPos, cur_ref = 0u, cur_cnt = 0u;
    bool live = false;                                        // this lane holds a ray whose walk is not over
    double r64[kRay64];
    TRay r;
    r.t = 0.0f; r.filt = r.tfilt = false; r.r64 = r64;
    bool more = true;                                         // warp-uniform: the source may still hold rays
    while (true) {
        const uint32_t idle = __ballot_sync(kFullMask, !live);
        if (more && __popc(idle) >= kRefillLanes) {
            bool got = false;
            more = job.refill(P, idle, got, r, r64);
            if (got) {
                sp = 0; tclosest = kFinf; closest_pos = kNoPos;                // raythread.cpp:204-205
                cur_ref = P.root_ref; cur_cnt = P.root_cnt;
                if (COUNT) lc.box++;
                live = root_accept(P, r);
                if (!live) job.finish(P, false, tclosest, closest_pos);      // missed the root box: found = false
            }
            continue;
        }
        if (idle == kFullMask) break;
        if (live) {
            bool need_pop = true;
            if (cur_cnt > 0) {
                for (uint32_t i = 0; i < cur_cnt; i++) {
                    uint32_t pos = cur_ref + i;
                    if (COUNT) lc.tri++;
                    const TriHit th = leaf_triangle<false, COUNT>(P, r, pos, lc);
                    if (th.hit) {
                        if (th.t > kEps) r.t = macro_min(r.t, th.t);               // bvh.cpp:161
                        if (r.t != kRayTInit && r.t < tclosest) {                  // bvh.cpp:212
                            closest_pos = pos; tclosest = r.t;
                        }
                    }
                }
            } else {
                CT_CHECK(cur_ref < P.n_pairs);
                DevPair32 pr;
                load_pair32(P.pairs32, cur_ref, pr);
                if (COUNT) lc.box += 2;
                bool hit_l, hit_r; float r_lo, r_hi;
                pair_accept<COUNT>(P, r, cur_ref, pr, hit_l, hit_r, r_lo, r_hi, lc);
                if (hit_l & hit_r) {
                    CT_CHECK(sp < kStackMax);
                    stk_ref[sp] = pr.r_ref; stk_cnt[sp] = pr.r_cnt;
                    stk_lo[sp] = r_lo; stk_hi[sp] = r_hi; stk_src[sp] = cur_ref;
                    sp++;
                }
                if (hit_l | hit_r) {
                    cur_ref = hit_l ? pr.l_ref : pr.r_ref; cur_cnt = hit_l ? pr.l_cnt : pr.r_cnt;
                    need_pop = false;
                }
            }
            if (need_pop) {
                live = false;
                while (sp > 0) {
                    --sp;
                    if (stk_lo[sp] >= r.t) continue;                          // the deferred `tmin < ray.t` of bvh.cpp:178
                    if (!(stk_hi[sp] < r.t)) {
                        if (COUNT) lc.box_exact++;
                        BoxTimes e = exact_child(P.pairs64, stk_src[sp], 1u, r.r64);
                        if (!(e.tmin < r.t)) continue;
                    }
                    cur_ref = stk_ref[sp]; cur_cnt = stk_cnt[sp]; live = true;
                    break;
                }
                if (!live) job.finish(P, r.t != kRayTInit, tclosest, closest_pos);      // raythread.cpp:227
            }
        }
    }
}

// The two early-exit walks.
//   kAnyHit    shadow rays (ray.t = 1e30f): only `found` is used (raythread.cpp:306), i.e. whether SOME triangle
//              reachable through accepted boxes has a barycentric pass with 1e-4 < t < 1e30 (SURVEY A7);
//   kFirstLine reflection rays (ray.t = 0, raythread.cpp:373): the first barycentric pass in DFS order becomes
//              closestIndex with tclosest = 0 (SURVEY 0.4).  The walks here keep the DFS order, so they find it on any
//              tree; the parked passes (overflow_merge, k_overflow_huge) take the LOWEST leaf position instead, which is
//              the same pass only where leaf positions increase along the DFS -- upload checks that (bvh_depth) and
//              never parks a first-line ray on a tree without it (first_line_budget).
// ray.t never changes before the exit, so the set of accepted boxes is fixed and the moment a leaf is tested
// cannot change the answer.  The loop therefore walks interior nodes only and DEFERS accepted leaves to a short
// list, in DFS order; the warp alternates between a walk phase and a leaf phase in which its lanes test their
// triangles together, oldest leaf first, instead of one lane at a time in the middle of the walk (measured: 4 of
// 32 lanes active in an inline leaf path, 16 in the leaf phase).  A leaf phase runs when some lane's list is full
// and after the walk; kFirstLine stops at the first pass of a phase (every leaf before it has been tested).
// WARP-SYNCHRONOUS like traverse_closest().  Returns kTravHit (kAnyHit: occluded; kFirstLine: always -- `found` is
// 0 != 1e30f, raythread.cpp:227 -- with closest_pos = kNoPos when nothing passed), kTravMiss or kTravOverBudget.
#ifndef CT_LEAF_LIST
#define CT_LEAF_LIST 8
#endif
constexpr int kLeafList = CT_LEAF_LIST;       // deferred leaves per lane before a leaf phase is forced
template <TraverseMode MODE, bool COUNT>
CT_DEV int traverse_early(const Params &P, const TRay &r, bool active, const uint32_t budget, float &tclosest, uint32_t &closest_pos, LocalCount &lc) {
    static_assert(MODE != kClosest, "closest-hit rays use traverse_closest");
    uint32_t stk_ref[kStackMax], stk_cnt[kStackMax];     // pushed right children
    uint32_t leaf_ref[kLeafList], leaf_cnt[kLeafList];   // deferred leaves, DFS order
    int sp = 0, nleaf = 0;
    uint32_t spent = 1u;
    uint32_t cur_ref = P.root_ref, cur_cnt = P.root_cnt;
    int state = 0;                                        // 1: nodes left to walk (cur_* pending); 0: walk finished
    int result = MODE == kFirstLine ? kTravHit : kTravMiss;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;      // "closestIndex = 0" default, resolved by the caller via pos_of_tri0
    const bool cons = r.filt & (P.nested != 0u);      // conservative box tests + verified candidates (see box_maybe)
    if (active) {
        if (COUNT) lc.box++;
        state = root_accept(P, r) ? 1 : 0;
    } else {
        result = kTravMiss;
    }
    while (true) {
        // ---- walk phase: one interior-node visit per walking lane and iteration; leaves go to the list
        while (__any_sync(kFullMask, (state == 1) & (nleaf < kLeafList))) {
            if ((state == 1) & (nleaf < kLeafList)) {
                bool descend = false;
                if (cur_cnt > 0) {
                    CT_CHECK(nleaf < kLeafList && cur_ref + cur_cnt <= P.n_tri);
                    leaf_ref[nleaf] = cur_ref; leaf_cnt[nleaf] = cur_cnt; nleaf++;
                    spent += cur_cnt;
                } else {
                    CT_CHECK(cur_ref < P.n_pairs);
                    DevPair32 pr;
                    load_pair32(P.pairs32, cur_ref, pr);
                    if (COUNT) lc.box += 2;
                    spent += 2u;
                    bool hit_l, hit_r;
                    if (cons) {
                        hit_l = box_maybe<MODE == kAnyHit>(r, pr.lmin, pr.lmax);
                        hit_r = box_maybe<MODE == kAnyHit>(r, pr.rmin, pr.rmax);
                    } else {
                        float r_lo, r_hi;
                        pair_accept<COUNT, MODE == kAnyHit>(P, r, cur_ref, pr, hit_l, hit_r, r_lo, r_hi, lc);
                    }
                    if (hit_l & hit_r) { CT_CHECK(sp < kStackMax); stk_ref[sp] = pr.r_ref; stk_cnt[sp] = pr.r_cnt; sp++; }
                    descend = hit_l | hit_r;
                    cur_ref = hit_l ? pr.l_ref : pr.r_ref; cur_cnt = hit_l ? pr.l_cnt : pr.r_cnt;
                }
                if (!descend) {
                    if (sp == 0) state = 0;
                    else { --sp; cur_ref = stk_ref[sp]; cur_cnt = stk_cnt[sp]; }
                }
                if (spent > budget) { result = kTravOverBudget; state = 0; nleaf = 0; }
            }
        }
        // ---- leaf phase: one triangle per lane and iteration, oldest leaf first
        int li = 0;
        uint32_t tri = 0;                                 // next triangle inside leaf li
        while (__any_sync(kFullMask, li < nleaf)) {
            if (li < nleaf) {
                const uint32_t pos = leaf_ref[li] + tri;
                if (COUNT) lc.tri++;
                const TriHit th = leaf_triangle<MODE == kAnyHit, COUNT>(P, r, pos, lc);
                bool done = MODE == kAnyHit ? (th.hit & (th.t > kEps) & (th.t < kRayTInit)) : th.hit;
                if (done & cons) done = candidate_reached(P, r, pos);     // the walk's box tests were only conservative
                if (done) {
                    if (MODE == kAnyHit) result = kTravHit;
                    else { closest_pos = pos; tclosest = 0.0f; }
                    state = 0; nleaf = 0;
                } else if (++tri == leaf_cnt[li]) { tri = 0; li++; }
            }
        }
        nleaf = 0;
        if (!__any_sync(kFullMask, state == 1)) break;
    }
    return result;
}

// The early-exit walks over the WIDE tree (DevWide, ct_layout.cuh), for rays whose box tests may be conservative
// (`cons` above: nested tree, no NaN among the slab quotients): every visit tests the kWide descendants kWideLevels
// levels down with box_maybe and skips the boxes in between -- a child's verdict implies its ancestors' -- so a ray
// descends the tree in 1 / kWideLevels of the dependent fetches and pays the loop's bookkeeping once per kWide boxes.
// Accepted children are pushed in reverse order and popped: the visit order is the reference's DFS order, deferred
// leaves reach the list in DFS order, and kFirstLine's "first pass of a leaf phase" is the DFS-first pass as in
// traverse_early (kAnyHit appends accepted leaves to the list at once; its answer does not depend on the order).
// A triangle that passes the exact test counts only if the reference's walk reaches its leaf (candidate_reached).
// WARP-SYNCHRONOUS, same contract as traverse_early; a stack that would overflow ends the walk as kTravOverBudget (the
// ray is parked and finished on the binary tree).
// Optional experiment (-DCT_TOP_SMEM=M, north_star: "BVH nodes staged through shared memory or TMA for the top levels"):
// the first M nodes of the wide tree -- they are numbered breadth first, so these are its top levels -- are copied into
// shared memory by one bulk-copy (TMA) instruction per CTA and the walk reads them from there.  Off by default: see the
// staging table in DESIGN.md 5.
#ifndef CT_TOP_SMEM
#define CT_TOP_SMEM 0
#endif
constexpr uint32_t kTopSmem = CT_TOP_SMEM;

// Stage the top of the wide tree: thread 0 arms an mbarrier with the byte count and issues one cp.async.bulk
// (global -> shared, completion on the mbarrier); everybody waits on the barrier's phase.  Returns the staged node count.
CT_DEV uint32_t stage_top_nodes(const Params &P, DevWide *top, unsigned long long *bar, uint32_t n_wide) {
    const uint32_t n_top = min(kTopSmem, n_wide);
    if (n_top == 0u) return 0u;
    const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(bar), dst_a = (uint32_t)__cvta_generic_to_shared(top);
    const uint32_t bytes = n_top * (uint32_t)sizeof(DevWide);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(dst_a), "l"(P.wide), "r"(bytes), "r"(bar_a) : "memory");
    }
    asm volatile("{\n .reg .pred p;\n WAIT_TOP:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n @p bra DONE_TOP;\n bra WAIT_TOP;\n DONE_TOP:\n}" ::"r"(bar_a) : "memory");
    return n_top;
}

// THE ANY-HIT WALK'S PER-LANE LISTS LIVE IN SHARED MEMORY (-DCT_SM_WALK=0: in local memory, as in round 1).  As local arrays
// the pending-children stack and the deferred-leaf list were more than half of the L1's sector traffic in every walk kernel
// (ncu, k_shadow: 137 M local sectors against 95 M global ones per launch; the lanes of a walking warp sit at different
// depths, so one STL / LDL touches up to 32 lines), every store went through to L2 (70 M write sectors = 2.2 GB per launch,
// 0.37 GB of it on to DRAM) and the lines shared the L1 with the tree.  In shared memory an access is one conflict-free
// wavefront whatever the lanes' indices (word w of thread t lives at sm[w * 128 + t]: bank = t mod 32), never leaves the SM
// and costs no tag look-up.  A lane keeps kSmStackWords stack entries there (one word each: an any-hit walk only pushes
// interior nodes) and its whole leaf list; deeper stack entries spill to a local array.  Shared memory is carved out of
// the L1, so less is more: measured on one box (dragon4k k_shadow / 66-light scene, ms): local lists 1.160 / 7.99;
// shared, stack 16 + 16 leaves (24 KB per CTA) 1.104 / 7.75; stack 8 + 12 leaves (16 KB) 1.112 / 7.14; stack 8 + 8 leaves
// 1.153 / 6.75 (a shorter leaf list also means earlier leaf phases: occluded rays leave sooner, lit ones pay more phases).
// The first-line walk (k_bounce) pushes leaves as well (two words per entry) and lost 2-6 % with its lists in shared
// memory at every size tried -- its rays are less coherent and want the L1 -- so it keeps local arrays.
#ifndef CT_SM_WALK
#define CT_SM_WALK 1
#endif
#ifndef CT_SM_STACK
#define CT_SM_STACK 8
#endif
#ifndef CT_ANY_LEAVES
#define CT_ANY_LEAVES 12
#endif
constexpr int kWideStack = 64;                 // pending children per lane: (kWide - 1) per level of the wide tree
#ifndef CT_LINE_LEAVES
#define CT_LINE_LEAVES (2 * kWide + 8)
#endif
constexpr int kWideLeaves = CT_LINE_LEAVES;     // deferred leaves per lane of a first-line walk; a visit may add kWide
constexpr int kAnyLeaves = CT_ANY_LEAVES;      // ... of an any-hit walk
constexpr int kSmStackWords = CT_SM_WALK ? CT_SM_STACK : 0;                 // shared-memory words per lane: stack ...
constexpr int kSmLeafWords = CT_SM_WALK ? 2 * kAnyLeaves : 0;               // ... and leaf list
constexpr int kWalkWords = CT_SM_WALK ? kSmStackWords + kSmLeafWords : 1;   // k_shadow declares walk_sm[kWalkWords * kBlockThreads]
template <TraverseMode MODE, bool COUNT>
CT_DEV int traverse_wide(const Params &P, const TRay &r, bool active, const uint32_t budget, float &tclosest, uint32_t &closest_pos, LocalCount &lc,
                         uint32_t *sm, const DevWide *top = nullptr, uint32_t n_top = 0u) {
    static_assert(MODE != kClosest, "closest-hit rays use traverse_closest");
    constexpr bool kUseSm = CT_SM_WALK && MODE == kAnyHit;                  // sm: this thread's column of walk_sm (any-hit walks only)
    constexpr int kLeaves = MODE == kAnyHit ? kAnyLeaves : kWideLeaves;
    constexpr int kSmEntries = kUseSm ? kSmStackWords : 0, kSmLeaves = kUseSm ? kAnyLeaves : 0;
    uint2 stk_spill[kWideStack - kSmEntries];             // pushed children (ref, cnt) beyond the shared-memory part
    uint2 leaf_spill[kLeaves - kSmLeaves + 1];            // deferred leaves (ref, cnt), DFS order
    uint32_t *const sm_leaf = sm + kSmStackWords * kBlockThreads;
    auto push = [&](int i, uint32_t ref, uint32_t cnt) {
        if (i < kSmEntries) sm[i * kBlockThreads] = ref;                    // (cnt = 0: interior nodes only)
        else stk_spill[i - kSmEntries] = make_uint2(ref, cnt);
    };
    auto pop = [&](int i) -> uint2 {
        if (i < kSmEntries) return make_uint2(sm[i * kBlockThreads], 0u);
        return stk_spill[i - kSmEntries];
    };
    auto leaf_put = [&](int i, uint32_t ref, uint32_t cnt) {
        if (i < kSmLeaves) { sm_leaf[(2 * i) * kBlockThreads] = ref; sm_leaf[(2 * i + 1) * kBlockThreads] = cnt; }
        else leaf_spill[i - kSmLeaves] = make_uint2(ref, cnt);
    };
    auto leaf_get = [&](int i) -> uint2 {
        if (i < kSmLeaves) return make_uint2(sm_leaf[(2 * i) * kBlockThreads], sm_leaf[(2 * i + 1) * kBlockThreads]);
        return leaf_spill[i - kSmLeaves];
    };
    int sp = 0, nleaf = 0;
    // a lane walks on while its list has room for a visit's worth of leaves; an any-hit walk may be told to use less of the list
    // (P.any_leaves: many-light scenes, where most rays are occluded and want their leaves tested early)
    const int leaf_room = (MODE == kAnyHit ? min(kLeaves, (int)P.any_leaves) : kLeaves) - kWide;
    uint32_t spent = 1u;
    uint32_t cur_ref = 0u, cur_cnt = P.root_cnt;          // wide node 0 = the root's descendants; a leaf root has no wide tree
    if (P.root_cnt > 0u) cur_ref = P.root_ref;
    int state = 0;                                        // 1: nodes left to walk (cur_* pending); 0: walk finished
    int result = MODE == kFirstLine ? kTravHit : kTravMiss;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;      // "closestIndex = 0" default, resolved by the caller via pos_of_tri0
    if (active) {
        if (COUNT) lc.box++;
        state = root_accept(P, r) ? 1 : 0;
    } else {
        result = kTravMiss;
    }
    while (true) {
        // ---- walk phase: one wide-node visit per walking lane and iteration; leaves go to the list
        while (__any_sync(kFullMask, (state == 1) & (nleaf <= leaf_room))) {
            if ((state == 1) & (nleaf <= leaf_room)) {
                if (cur_cnt > 0u) {                       // a leaf that came off the stack (or a leaf root)
                    leaf_put(nleaf, cur_ref, cur_cnt); nleaf++;
                    spent += cur_cnt;
                } else {
                    const float4 *q = reinterpret_cast<const float4 *>(P.wide + cur_ref);
                    const bool staged = kTopSmem > 0u && cur_ref < n_top;             // (generic loads below when the experiment is on)
                    if (staged) q = reinterpret_cast<const float4 *>(top + cur_ref);
                    if (COUNT) lc.box += kWide;
                    spent += (uint32_t)kWide;
                    if (sp > kWideStack - kWide) { result = kTravOverBudget; state = 0; nleaf = 0; sp = 0; }
                    else {
#pragma unroll
                        for (int e = kWide - 1; e >= 0; e--) {             // reverse: the first accepted child is popped first
                            float4 a; uint4 b;
                            if (kTopSmem > 0u) { a = q[2 * e]; b = *reinterpret_cast<const uint4 *>(q + 2 * e + 1); }
                            else ldg256(q + 2 * e, a, b);
                            const float bmin[3] = {a.x, a.y, a.z}, bmax[3] = {a.w, __uint_as_float(b.x), __uint_as_float(b.y)};
                            const bool hit = box_maybe<MODE == kAnyHit>(r, bmin, bmax);
                            if (MODE == kAnyHit) {
                                const bool is_leaf = b.w > 0u;
                                if (hit & is_leaf) { leaf_put(nleaf, b.z, b.w); nleaf++; spent += b.w; }
                                if (hit & !is_leaf) { push(sp, b.z, 0u); sp++; }
                            } else {
                                if (hit) { push(sp, b.z, b.w); sp++; }
                            }
                        }
                    }
                }
                if (state == 1) {
                    if (sp == 0) state = 0;
                    else { --sp; const uint2 t = pop(sp); cur_ref = t.x; cur_cnt = t.y; }
                }
                if (spent > budget) { result = kTravOverBudget; state = 0; nleaf = 0; }
            }
        }
        // ---- leaf phase: one triangle per lane and iteration, oldest leaf first
        int li = 0;
        uint32_t tri = 0;                                 // next triangle inside leaf li
        while (__any_sync(kFullMask, li < nleaf)) {
            if (li < nleaf) {
                const uint2 lf = leaf_get(li);
                const uint32_t pos = lf.x + tri;
                if (COUNT) lc.tri++;
                const TriHit th = leaf_triangle<MODE == kAnyHit, COUNT>(P, r, pos, lc);
                bool done = MODE == kAnyHit ? (th.hit & (th.t > kEps) & (th.t < kRayTInit)) : th.hit;
                if (done) done = candidate_reached(P, r, pos);        // the walk's box tests were only conservative
                if (done) {
                    if (MODE == kAnyHit) result = kTravHit;
                    else { closest_pos = pos; tclosest = 0.0f; }
                    state = 0; nleaf = 0;
                } else if (++tri == lf.y) { tri = 0; li++; }
            }
        }
        nleaf = 0;
        if (!__any_sync(kFullMask, state == 1)) break;
    }
    return result;
}

// IntersectBVHClosest over the wide tree.  On a nested tree the closest-hit walk is, like the early-exit walks, a matter of
// its LEAVES only: with ray.t only ever decreasing,  tmin(ancestor) <= tmin(leaf) < ray.t(at the leaf's visit) <= ray.t(at
// the ancestor's visit),  so the reference visits a leaf exactly when the leaf's own box passes IntersectAABB against the
// ray.t of that moment -- i.e. the reference's result is that of scanning the leaves in DFS order, testing each leaf's own
// box against the current ray.t and, where it passes, its triangles in order (bvh.cpp:198-222).  So:
//   * the walk enumerates candidate leaves in DFS order with the conservative box_maybe against whatever ray.t it holds
//     at the time -- never smaller than the reference's at that node, because the leaves processed so far all precede the
//     node in DFS order -- hence a superset of the leaves the reference visits, in the reference's order;
//   * leaves are deferred to the list and processed in the leaf phase, oldest first: the exact slab test of the leaf's
//     own box (certified bracket, fp64 when undecided) against the CURRENT ray.t, then its triangles in order with the
//     reference's update rules.
// Same hits, same order, same ray.t / tclosest / closestIndex as traverse_closest; rays that do not allow conservative
// tests (and walks whose stack would overflow) take traverse_closest.  WARP-SYNCHRONOUS.
// How long the walk runs ahead of the leaf tests decides how stale the ray.t it prunes with is (a closest-hit walk lives on
// pruning): a lane defers at most kClosestLeaves leaves, and a leaf phase starts as soon as kClosestLanes lanes hold one.
#ifndef CT_CLOSEST_LEAVES
#define CT_CLOSEST_LEAVES 1
#endif
#ifndef CT_CLOSEST_LANES
#define CT_CLOSEST_LANES 24
#endif
constexpr int kClosestLeaves = CT_CLOSEST_LEAVES, kClosestLanes = CT_CLOSEST_LANES;
template <bool COUNT>
CT_DEV int traverse_wide_closest(const Params &P, TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc) {
    uint2 stk[kWideStack];
    uint2 leaf[kClosestLeaves];
    int sp = 0, nleaf = 0;
    uint32_t cur_ref = 0u, cur_cnt = P.root_cnt;
    if (P.root_cnt > 0u) cur_ref = P.root_ref;
    int state = 0;
    bool overflow = false;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;
    if (active) {
        if (COUNT) lc.box++;
        state = root_accept(P, r) ? 1 : 0;
    }
    while (true) {
        // ---- walk phase: candidate leaves in DFS order
        while (__any_sync(kFullMask, (state == 1) & (nleaf < kClosestLeaves)) && __popc(__ballot_sync(kFullMask, nleaf > 0)) < kClosestLanes) {
            if ((state == 1) & (nleaf < kClosestLeaves)) {
                if (cur_cnt > 0u) {
                    leaf[nleaf] = make_uint2(cur_ref, cur_cnt); nleaf++;
                } else if (sp > kWideStack - kWide) {
                    overflow = true; state = 0; nleaf = 0; sp = 0;
                } else {
                    const float4 *q = reinterpret_cast<const float4 *>(P.wide + cur_ref);
                    if (COUNT) lc.box += kWide;
#pragma unroll
                    for (int e = kWide - 1; e >= 0; e--) {                 // reverse: the first accepted child is popped first
                        float4 a; uint4 b;
                        ldg256(q + 2 * e, a, b);
                        const float bmin[3] = {a.x, a.y, a.z}, bmax[3] = {a.w, __uint_as_float(b.x), __uint_as_float(b.y)};
                        if (box_maybe<false>(r, bmin, bmax)) { stk[sp] = make_uint2(b.z, b.w); sp++; }
                    }
                }
                if (state == 1) {
                    if (sp == 0) state = 0;
                    else { --sp; const uint2 t = stk[sp]; cur_ref = t.x; cur_cnt = t.y; }
                }
            }
        }
        // ---- leaf phase: the deferred leaves in order; per iteration a lane either opens its next leaf (the exact test of
        // the leaf's own box against the current ray.t) or tests one triangle of the open leaf
        int li = 0;
        uint32_t tri = 0;
        bool open = false;
        while (__any_sync(kFullMask, li < nleaf)) {
            if (li < nleaf) {
                const uint2 lf = leaf[li];
                if (!open) {
                    const uint32_t code = __ldg(P.tri_parent + lf.x);
                    bool acc;
                    if (code == kNoPos) acc = true;                    // the root itself: accepted before the walk (nothing has changed ray.t since)
                    else {
                        const uint32_t pid = code >> 1, side = code & 1u;
                        const float4 *q = reinterpret_cast<const float4 *>(P.pairs32 + pid);
                        const float4 x = __ldg(q + side), y = __ldg(q + 1 + side);      // left: floats 0..5, right: floats 6..11
                        float bmin[3], bmax[3];
                        if (side == 0u) { bmin[0] = x.x; bmin[1] = x.y; bmin[2] = x.z; bmax[0] = x.w; bmax[1] = y.x; bmax[2] = y.y; }
                        else { bmin[0] = x.z; bmin[1] = x.w; bmin[2] = y.x; bmax[0] = y.y; bmax[1] = y.z; bmax[2] = y.w; }
                        const BoxBracket bb = box_filter(r, bmin, bmax);
                        const bool no = bracket_geom_no(bb) | bracket_t_no(bb, r.t), yes = bracket_geom_yes(bb) & bracket_t_yes(bb, r.t);
                        acc = yes;
                        if (!(no | yes)) {
                            if (COUNT) lc.box_exact++;
                            acc = box_accept(exact_child(P.pairs64, pid, side, r.r64), r.t);
                        }
                    }
                    if (COUNT) lc.box++;
                    if (acc) { open = true; tri = 0; } else li++;
                } else {
                    const uint32_t pos = lf.x + tri;
                    if (COUNT) lc.tri++;
                    const TriHit th = leaf_triangle<false, COUNT>(P, r, pos, lc);
                    if (th.hit) {
                        if (th.t > kEps) r.t = macro_min(r.t, th.t);               // bvh.cpp:161
                        if (r.t != kRayTInit && r.t < tclosest) {                  // bvh.cpp:212
                            closest_pos = pos; tclosest = r.t;
                        }
                    }
                    if (++tri == lf.y) { open = false; li++; }
                }
            }
        }
        nleaf = 0;
        if (!__any_sync(kFullMask, state == 1)) break;
    }
    if (!active) return kTravMiss;
    if (overflow) return kTravOverBudget;
    return r.t != kRayTInit ? kTravHit : kTravMiss;
}

// IntersectBVHClosest as an ORDER-FREE search (primary rays, ray.t = 1e30f).  On a nested tree the reference tests a triangle
// iff its LEAF's own box passes IntersectAABB against the ray.t of that moment (see traverse_wide_closest).  Let G be the
// triangles with a barycentric pass and 1e-4 < t < 1e30 whose leaf box passes the two conditions that do not involve ray.t,
// m = min t over G, and sigma the ray's slop bound (tray_nearest_setup:  tmin(leaf of Z) <= t_Z + sigma  for every Z).  Then
//   * ray.t never drops below m; the first triangle with t = m is tested unless ray.t <= tmin(its leaf) <= m + sigma by
//     then -- either way the walk ends with ray.t <= m + sigma;
//   * a triangle with t > tau changes the fate of one with t <= tau only by lowering ray.t to a value that blocks the
//     latter's leaf, i.e. only if  tmin(that leaf) >= t > tau.
// So with S = { Z in G : t_Z <= m + sigma }:  if every member of S has tmin(leaf) <= m + sigma, nothing outside S can block
// a member of S, a tested member of S lowers ray.t below anything outside S, and replaying the reference's update rules
// (bvh.cpp:161, 178, 212) over S alone, in leaf-position order (= the reference's test order), gives the reference's
// ray.t, tclosest and closestIndex bit for bit.  Finding S needs no particular order: the walk keeps best = min t so far
// and prunes a box only when the LOWER end of its near bracket is >= best + 2 sigma: every triangle Z below it has
// t_Z >= tmin(leaf of Z) - sigma >= tmin(box) - sigma >= best + sigma >= m + sigma (boxes are nested, best >= m; sigma
// carries slack, so the inequality is strict) and is not in S.  Each barycentric pass within best + sigma becomes a candidate once the exact fp64 test of its own leaf box confirms membership in G (that test also
// yields the reference's tmin for the replay).  The rare leftovers -- more than kNearCand candidates, a member of S whose
// leaf starts beyond m + sigma, t >= FINF (raythread.cpp:204's tclosest quirk), a full stack -- return kTravOverBudget
// and take traverse_closest.  The argument is checked on the CPU by tests/test_free_closest_prototype.py.
// What the freedom buys: conservative one-sided box tests over the wide tree (half the FMAs of the certified brackets, half
// the dependent fetches, no fp64 fallback), leaves tested by the warp together, and a walk that may be cut short.
// WARP-SYNCHRONOUS, same contract as traverse_closest for the rays it decides.
#ifndef CT_NEAR_LEAVES
#define CT_NEAR_LEAVES 1
#endif
#ifndef CT_NEAR_LANES
#define CT_NEAR_LANES 24
#endif
constexpr int kNearLeaves = CT_NEAR_LEAVES, kNearLanes = CT_NEAR_LANES, kNearCand = 4;      // kNearLeaves = 0: leaves are tested on the spot
constexpr int kNearLeavesCap = kNearLeaves > 0 ? kNearLeaves : 1;
template <bool COUNT>
CT_DEV int traverse_wide_nearest(const Params &P, const TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc) {
    uint2 stk[kWideStack];
    float stk_near[kWideStack];                           // lower end of the pushed child's near bracket
    uint2 leaf[kNearLeavesCap];
    float cand_t[kNearCand], cand_tmin[kNearCand];
    uint32_t cand_pos[kNearCand], cand_code[kNearCand];
    int sp = 0, nleaf = 0, ncand = 0;
    float best = kRayTInit, band = kRayTInit, thr = kRayTInit;     // band >= best + sigma, thr >= best + 2 sigma
    uint32_t cur_ref = 0u, cur_cnt = P.root_cnt;
    if (P.root_cnt > 0u) cur_ref = P.root_ref;
    int state = 0;
    bool undecided = false;
    tclosest = kFinf;          // raythread.cpp:204
    closest_pos = kNoPos;
    if (active) {
        if (COUNT) lc.box++;
        state = root_accept(P, r) ? 1 : 0;
    }
    auto test_triangle = [&](uint32_t pos) {
        if (COUNT) lc.tri++;
        const TriHit th = leaf_triangle<false, COUNT>(P, r, pos, lc);
        if (th.hit & (th.t > kEps) & (th.t < kRayTInit)) {                     // would lower a ray.t of 1e30f (bvh.cpp:161)
            if (!(th.t < kFinf)) undecided = true;
            else if (th.t <= band) {
                const uint32_t code = __ldg(P.tri_parent + pos);               // the triangle's leaf: 2 * pair + side
                if (COUNT) lc.box_exact++;
                const BoxTimes e = code == kNoPos ? box_times(r.r64, P.root_min, P.root_max) : exact_child(P.pairs64, code >> 1, code & 1u, r.r64);
                if ((e.tmax >= e.tmin) & (e.tmax > 0.0f)) {                    // the leaf is one the reference can reach: Z is in G
                    if (th.t < best) { best = th.t; band = __fadd_ru(best, r.sg); thr = __fadd_ru(band, r.sg); }
                    if (ncand == kNearCand) {                                  // drop what has fallen out of the band
                        int k = 0;
                        for (int j = 0; j < kNearCand; j++)
                            if (cand_t[j] <= band) { cand_t[k] = cand_t[j]; cand_tmin[k] = cand_tmin[j]; cand_pos[k] = cand_pos[j]; cand_code[k] = cand_code[j]; k++; }
                        ncand = k;
                    }
                    if (ncand == kNearCand) undecided = true;
                    else { cand_t[ncand] = th.t; cand_tmin[ncand] = e.tmin; cand_pos[ncand] = pos; cand_code[ncand] = code; ncand++; }
                }
            }
        }
    };
    while (true) {
        // ---- walk phase: one wide-node visit per walking lane and iteration
        while (__any_sync(kFullMask, (state == 1) & (nleaf < kNearLeavesCap)) && __popc(__ballot_sync(kFullMask, nleaf > 0)) < kNearLanes) {
            if ((state == 1) & (nleaf < kNearLeavesCap)) {
                if (cur_cnt > 0u) {
                    if (kNearLeaves == 0) {                                 // on the spot
                        for (uint32_t i = 0; i < cur_cnt; i++) test_triangle(cur_ref + i);
                        if (undecided) { state = 0; sp = 0; }
                    }
                    else { leaf[nleaf] = make_uint2(cur_ref, cur_cnt); nleaf++; }
                } else if (sp > kWideStack - kWide) {
                    undecided = true; state = 0; nleaf = 0; sp = 0;
                } else {
                    const float4 *q = reinterpret_cast<const float4 *>(P.wide + cur_ref);
                    if (COUNT) lc.box += kWide;
#pragma unroll
                    for (int e = kWide - 1; e >= 0; e--) {                 // reverse: the first accepted child is popped first
                        float4 a; uint4 b;
                        ldg256(q + 2 * e, a, b);
                        const float bmax1 = __uint_as_float(b.x), bmax2 = __uint_as_float(b.y);
                        const bool px = r.rdf[0] > 0.0f, py = r.rdf[1] > 0.0f, pz = r.rdf[2] > 0.0f;
                        const float n0 = __fmaf_rd(px ? a.x : a.w, r.rdf[0], r.cl[0]), f0 = __fmaf_ru(px ? a.w : a.x, r.rdf[0], r.cu[0]);
                        const float n1 = __fmaf_rd(py ? a.y : bmax1, r.rdf[1], r.cl[1]), f1 = __fmaf_ru(py ? bmax1 : a.y, r.rdf[1], r.cu[1]);
                        const float n2 = __fmaf_rd(pz ? a.z : bmax2, r.rdf[2], r.cl[2]), f2 = __fmaf_ru(pz ? bmax2 : a.z, r.rdf[2], r.cu[2]);
                        const float near_lo = fmaxf(fmaxf(n0, n1), n2), far_hi = fminf(fminf(f0, f1), f2);      // box_maybe's brackets
                        const bool no = (far_hi < near_lo) | (far_hi <= 0.0f) | (near_lo >= thr);
                        if (!no) { stk[sp] = make_uint2(b.z, b.w); stk_near[sp] = near_lo; sp++; }
                    }
                }
                if (state == 1) {
                    state = 0;
                    while (sp > 0) {                                       // best may have dropped since the child was pushed
                        --sp;
                        if (stk_near[sp] >= thr) continue;
                        const uint2 t = stk[sp]; cur_ref = t.x; cur_cnt = t.y; state = 1;
                        break;
                    }
                }
            }
        }
        // ---- leaf phase: one triangle per lane and iteration
        int li = 0;
        uint32_t tri = 0;
        while (__any_sync(kFullMask, li < nleaf)) {
            if (li < nleaf) {
                const uint2 lf = leaf[li];
                const uint32_t pos = lf.x + tri;
                test_triangle(pos);
                if (++tri == lf.y) { tri = 0; li++; }
            }
        }
        nleaf = 0;
        if (undecided) { state = 0; sp = 0; }
        if (!__any_sync(kFullMask, state == 1)) break;
    }
    if (!active) return kTravMiss;
    if (undecided) return kTravOverBudget;
    if (best == kRayTInit) return kTravMiss;                                           // ray.t never changes
    // ---- S, its precondition, and the replay in leaf-position order
    int n = 0;
    for (int j = 0; j < ncand; j++)
        if (cand_t[j] <= band) { cand_t[n] = cand_t[j]; cand_tmin[n] = cand_tmin[j]; cand_pos[n] = cand_pos[j]; cand_code[n] = cand_code[j]; n++; }
    for (int j = 0; j < n; j++) if (!(cand_tmin[j] <= band)) return kTravOverBudget;
    for (int j = 1; j < n; j++) {
        const float zt = cand_t[j], zm = cand_tmin[j]; const uint32_t zp = cand_pos[j], zc = cand_code[j];
        int k = j;
        while (k > 0 && cand_pos[k - 1] > zp) { cand_t[k] = cand_t[k - 1]; cand_tmin[k] = cand_tmin[k - 1]; cand_pos[k] = cand_pos[k - 1]; cand_code[k] = cand_code[k - 1]; k--; }
        cand_t[k] = zt; cand_tmin[k] = zm; cand_pos[k] = zp; cand_code[k] = zc;
    }
    float rt = kRayTInit;
    uint32_t entered = 0xfffffffeu;                                                    // (no leaf has this code)
    for (int j = 0; j < n; j++) {
        if (cand_code[j] != entered) {                                                 // the box is tested once per leaf visit
            if (!(cand_tmin[j] < rt)) continue;                                        // bvh.cpp:178, the leaf's own box
            entered = cand_code[j];
        }
        rt = macro_min(rt, cand_t[j]);                                                 // bvh.cpp:161
        if (rt != kRayTInit && rt < tclosest) { closest_pos = cand_pos[j]; tclosest = rt; }   // bvh.cpp:212
    }
    return rt != kRayTInit ? kTravHit : kTravMiss;
}

// The closest-hit walk for every lane's ray: over the wide tree where the ray allows conservative box tests, the binary
// walk with the reference's verdict at every box otherwise.
// Measured (DESIGN.md 5): the wide closest-hit walk is 7 % faster than the binary one on the dragon-class frame, 8 % slower
// on the bunny and 30 % slower on scene_import.json (leaves of up to 54 triangles) -- a closest-hit walk wants its leaves
// tested at once, which is what the binary walk does.  It is therefore an experiment: -DCT_WIDE_CLOSEST=1 switches it on.
#ifndef CT_WIDE_CLOSEST
#define CT_WIDE_CLOSEST 0
#endif
#ifndef CT_CONS_CLOSEST
#define CT_CONS_CLOSEST 0            // 1: the ordered closest-hit walk tests interior boxes conservatively and opens leaves exactly (traverse_closest_cons) -- measured slower, DESIGN.md 5
#endif
#ifndef CT_NEAREST
#define CT_NEAREST 0                 // 1: primary rays take the order-free walk (traverse_wide_nearest) where the ray allows it -- measured slower, DESIGN.md 5
#endif
template <bool COUNT, bool BUDGETED = false>
CT_DEV int traverse_closest_any(const Params &P, TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc, uint32_t *sm = nullptr,
                                const uint32_t budget = 0xffffffffu) {
    if (CT_NEAREST) {
        // r.sg > 0: tray_nearest_setup found the ray within the limits of the slop analysis (and r.filt); ray.t must be 1e30f
        const bool fr = active & (r.sg > 0.0f) & (r.t == kRayTInit) & (P.nested != 0u) & (P.wide != nullptr);
        int res = traverse_wide_nearest<COUNT>(P, r, fr, tclosest, closest_pos, lc);
        const bool ordered = active & (!fr | (res == kTravOverBudget));
        if (__any_sync(kFullMask, ordered)) {                          // the ordered walk decides the rest
            float tc2; uint32_t pos2;
            const int res2 = traverse_closest<COUNT>(P, r, ordered, tc2, pos2, lc);
            if (ordered) { res = res2; tclosest = tc2; closest_pos = pos2; }
        }
        return res;
    }
    if (CT_CONS_CLOSEST) {
        const bool cons = active & r.filt & (P.nested != 0u);
        int res = traverse_closest_cons<COUNT>(P, r, cons, tclosest, closest_pos, lc);
        const bool rest = active & !cons;
        if (__any_sync(kFullMask, rest)) {                             // zero direction components, trees that are not nested
            float tc2; uint32_t pos2;
            const int res2 = traverse_closest<COUNT>(P, r, rest, tc2, pos2, lc);
            if (rest) { res = res2; tclosest = tc2; closest_pos = pos2; }
        }
        return res;
    }
    if (!CT_WIDE_CLOSEST) return traverse_closest<COUNT, BUDGETED>(P, r, active, tclosest, closest_pos, lc, sm, budget);
    const bool cons = r.filt & (P.nested != 0u) & (P.wide != nullptr);
    const float t0 = r.t;
    int res = traverse_wide_closest<COUNT>(P, r, active & cons, tclosest, closest_pos, lc);
    const bool binary = active & (!cons | (res == kTravOverBudget));
    if (__any_sync(kFullMask, binary)) {
        float tc2; uint32_t pos2;
        if (binary) r.t = t0;                                          // (a walk given up half way starts over)
        const int res2 = traverse_closest<COUNT>(P, r, binary, tc2, pos2, lc);
        if (binary) { res = res2; tclosest = tc2; closest_pos = pos2; }
    }
    return res;
}

// An early-exit walk for every lane's ray: over the wide tree where the ray allows conservative box tests, with the
// reference's exact verdicts at every box of the binary tree otherwise (zero direction components, non-nested trees).
template <TraverseMode MODE, bool COUNT>
CT_DEV int traverse_early_any(const Params &P, const TRay &r, bool active, const uint32_t budget, float &tclosest, uint32_t &closest_pos, LocalCount &lc,
                              uint32_t *sm, const DevWide *top = nullptr, uint32_t n_top = 0u) {
    const bool cons = r.filt & (P.nested != 0u) & (P.wide != nullptr);
    int res = traverse_wide<MODE, COUNT>(P, r, active & cons, budget, tclosest, closest_pos, lc, sm, top, n_top);
    // the binary walk for the other rays, and for rays that may not be parked (no budget) whose wide stack overflowed
    const bool binary = active & (!cons | ((res == kTravOverBudget) & (budget == 0xffffffffu)));
    if (__any_sync(kFullMask, binary)) {
        float tc2; uint32_t pos2;
        const int res2 = traverse_early<MODE, COUNT>(P, r, binary, budget, tc2, pos2, lc);
        if (binary) { res = res2; tclosest = tc2; closest_pos = pos2; }
    }
    return res;
}

}  // namespace
