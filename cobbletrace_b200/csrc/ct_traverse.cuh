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

// 32 bytes per lane in ONE load instruction (ld.global.nc.v8 -> LDG.E.256, new with sm_100): a whole child of a wide
// node, half a child pair.  The lanes of a walking warp read 32 different records, so every load instruction costs the
// L1 one tag look-up per lane whatever its width -- the walks are bound by exactly that (l1tex throughput 79 % of peak in
// k_shadow) -- and a 256-bit load halves the look-ups per record.  p: 32-byte aligned.
CT_DEV void ldg256(const void *p, float4 &a, uint4 &b) {
    uint32_t x0, x1, x2, x3;
    asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(x0), "=r"(x1), "=r"(x2), "=r"(x3), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
    a = make_float4(__uint_as_float(x0), __uint_as_float(x1), __uint_as_float(x2), __uint_as_float(x3));
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
// `spill` is never dereferenced: no push happens at sp < 0.  That branch is kept on purpose: until the compiler proves it dead,
// its store through an unknown pointer stops LLVM from hoisting Params' fields out of the walk loop into registers, so ptxas
// reads them from the constant bank at each use.  Without it k_primary / k_primary_long / k_primary_split compile to other
// SASS, k_primary_long<false> with 16 more bytes of stack and more spills, and (with PrimaryJob::refill's plain `lane`) the
// dragon 4K stages measured slower on a B200 at 1000 W: k_primary 1.546 -> 1.553 ms, k_primary_long 0.395 -> 0.414 ms.
template <bool COUNT, bool BUDGETED = false>
CT_DEV int traverse_closest(const Params &P, TRay &r, bool active, float &tclosest, uint32_t &closest_pos, LocalCount &lc,
                            uint32_t *spill = nullptr, const uint32_t budget = 0xffffffffu) {
    // stack entry = a pushed right child: (ref, cnt), the bracket of its tmin and its parent pair (to find its fp64
    // bounds again when the bracket cannot decide)
    uint32_t stk_ref[kStackMax], stk_cnt[kStackMax], stk_src[kStackMax];
    float stk_lo[kStackMax], stk_hi[kStackMax];
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
                if (BUDGETED && ++visits > budget) { over = true; live = false; continue; }      // a long walk: the caller parks the ray (k_primary<COUNT, true>)
                DevPair32 pr;
                load_pair32(P.pairs32, cur_ref, pr);
                if (COUNT) lc.box += 2;
                bool hit_l, hit_r; float r_lo, r_hi;
                pair_accept<COUNT>(P, r, cur_ref, pr, hit_l, hit_r, r_lo, r_hi, lc);
                if (hit_l & hit_r) {
                    CT_CHECK(sp < kStackMax);
                    if (sp < 0) {
                        for (int w = 0; w < 5; w++) spill[(5 * sp + w) * kBlockThreads] = 0u;
                    } else {
                        stk_ref[sp] = pr.r_ref; stk_cnt[sp] = pr.r_cnt; stk_lo[sp] = r_lo; stk_hi[sp] = r_hi; stk_src[sp] = cur_ref;
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
                    if (stk_lo[sp] >= r.t) continue;                          // the deferred `tmin < ray.t` of bvh.cpp:178
                    if (!(stk_hi[sp] < r.t)) {
                        if (COUNT) lc.box_exact++;
                        BoxTimes e = exact_child(P.pairs64, stk_src[sp], 1u, r.r64);
                        if (!(e.tmin < r.t)) continue;
                    }
                    cur_ref = stk_ref[sp]; cur_cnt = stk_cnt[sp]; live = true;
                    break;
                }
            }
        }
    }
    if (!active) return kTravMiss;
    if (BUDGETED && over) return kTravOverBudget;          // given up after `budget` pair visits: ray.t, tclosest, closest_pos are those of a walk half done
    return r.t != kRayTInit ? kTravHit : kTravMiss;
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
//
// THE ANY-HIT WALK'S PER-LANE LISTS LIVE IN SHARED MEMORY.  As local arrays (round 1)
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
constexpr int kSmStackWords = CT_SM_STACK;                   // shared-memory words per lane: stack ...
constexpr int kSmLeafWords = 2 * kAnyLeaves;                // ... and leaf list
constexpr int kWalkWords = kSmStackWords + kSmLeafWords;    // k_shadow declares walk_sm[kWalkWords * kBlockThreads]
template <TraverseMode MODE, bool COUNT>
CT_DEV int traverse_wide(const Params &P, const TRay &r, bool active, const uint32_t budget, float &tclosest, uint32_t &closest_pos, LocalCount &lc,
                         uint32_t *sm) {
    static_assert(MODE != kClosest, "closest-hit rays use traverse_closest");
    constexpr bool kUseSm = MODE == kAnyHit;                                // sm: this thread's column of walk_sm (any-hit walks only)
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
                    if (COUNT) lc.box += kWide;
                    spent += (uint32_t)kWide;
                    if (sp > kWideStack - kWide) { result = kTravOverBudget; state = 0; nleaf = 0; sp = 0; }
                    else {
#pragma unroll
                        for (int e = kWide - 1; e >= 0; e--) {             // reverse: the first accepted child is popped first
                            float4 a; uint4 b;
                            ldg256(q + 2 * e, a, b);
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

// An early-exit walk for every lane's ray: over the wide tree where the ray allows conservative box tests, with the
// reference's exact verdicts at every box of the binary tree otherwise (zero direction components, non-nested trees).
template <TraverseMode MODE, bool COUNT>
CT_DEV int traverse_early_any(const Params &P, const TRay &r, bool active, const uint32_t budget, float &tclosest, uint32_t &closest_pos, LocalCount &lc,
                              uint32_t *sm) {
    const bool cons = r.filt & (P.nested != 0u) & (P.wide != nullptr);
    int res = traverse_wide<MODE, COUNT>(P, r, active & cons, budget, tclosest, closest_pos, lc, sm);
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
