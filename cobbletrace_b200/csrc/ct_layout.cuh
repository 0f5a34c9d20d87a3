// ct_layout.cuh -- constants, the device-side scene layout, per-tile scheduling state and the kernel parameter block.
// Part of the single translation unit ct_gpu.cu (everything lives in its anonymous namespace).
#pragma once

#include <cstdint>

#include "../../include/ct_gpu.h"
#include "ct_exact.cuh"

namespace {

using namespace ct;

constexpr int kStackMax = 96;        // DFS stack entries per ray (tree depth limit, checked at upload)
constexpr int kMaxDevices = 16;
constexpr int kBlockThreads = 128;   // 4 warps per CTA
#ifndef CT_MIN_BLOCKS
#define CT_MIN_BLOCKS 6
#endif
constexpr int kMinBlocks = CT_MIN_BLOCKS;   // traversal kernels: resident CTAs per SM the register allocation must allow
constexpr int kOvfThreads = 256;     // k_overflow CTA
constexpr int kMaxLaunches = 80;     // launches of one tile (work cursors / stage events)
constexpr uint32_t kNoPos = 0xffffffffu;
constexpr uint32_t kNoReuse = 0x80000000u;      // parent_q flag: the reflection ray's direction is not finite (0 * direction would not be 0)
constexpr int kCursorStride = 16;    // unsigned long longs between the two chunk cursors of a shared frame (128 bytes)
// Slots a warp takes from the tile's cursor at a time: 32 = one 8x4 pixel block, one ray per lane.  When the cursor is
// another GPU's memory, 64 would halve the NVLink round trips, but a kernel ends with its slowest warp and a warp's
// chunk is walked one ray per lane at a time: measured on dragon 4K, 2 / 4 GPUs: 4.10 / 2.49 ms with 64 against
// 4.01 / 2.36 ms with 32 (option "shared_chunk_shift" for experiments).
constexpr uint32_t kChunkLocalShift = 5;
constexpr uint32_t kChunkSharedShift = 5;
constexpr uint32_t kChunkMaxShift = 6;
constexpr uint32_t kChunkMax = 1u << kChunkMaxShift;
constexpr uint32_t kDefaultBudget = 384;    // node visits + triangle tests before a ray is parked for k_overflow
// Pair visits after which a primary ray's walk is given up and the ray parked: k_primary_long walks the parked rays again, from
// the start, in warps that hold long walks only (option "primary_budget").  The mean primary walk of the dragon-class frame is 26
// pair visits, 2.7 % of the rays need more than 64 and the longest ~300 -- and while one lane finishes such a walk the other 31
// idle: cutting every walk at 64 visits (timing experiment, wrong pixels) took 21 % off k_primary.  But a lone walk advances at
// ~1 us per DEPENDENT pair visit whoever its neighbours are, so the second kernel cannot end before its longest walk has:
// measured k_primary 1.64 -> 1.31 ms + k_primary_long 0.55 ms at a budget of 64 (0.41 -> 0.24 + 0.31 ms for one rank's 1/8 share).
// OFF by default (0); only splitting a long walk across lanes can shorten it (DESIGN.md 8).
constexpr uint32_t kDefaultPrimaryBudget = 0;

// ---- device-side scene layout (SoA arrays in HBM, uploaded once) -----------------------------------
// The BVH is stored per INTERIOR node as the pair of its two children (bvh.cpp:89-97 allocates them adjacently
// and the traversal always needs both).  A child is described by (ref, cnt): cnt > 0 -> leaf holding triangles
// [ref, ref + cnt) of the leaf-ordered triangle array; cnt == 0 -> interior, ref = its own pair index.
struct __align__(16) DevPair32 {     // 64 B = two 32-B sectors: what the certified fp32 filter reads
    float lmin[3], lmax[3], rmin[3], rmax[3];    // float(bounds), round to nearest
    uint32_t l_ref, l_cnt, r_ref, r_cnt;
};
struct __align__(16) DevPair64 {     // 96 B: the reference's fp64 bounds, read only when the filter cannot decide
    double lmin[3], lmax[3], rmin[3], rmax[3];
};
struct __align__(16) DevTri {        // 80 B, stored in LEAF order (position = slot in bvh indexes[])
    double p1[3], e1[3], e2[3];      // e1 = p2-p1, e2 = p3-p1 (bvh.cpp:148-149, raythread.cpp:337-338)
    uint32_t orig, pad;              // original triangle id (= closestIndex of the reference)
};
struct __align__(16) DevTri32 {      // 48 B, same order: what the certified fp32 triangle filter reads
    float p1[3], k3;                 // k3 = max|p1_i| rounded up
    float e1[3], k1;                 // k1 = max|e1_i| rounded up (NaN: magnitudes outside the filter's range)
    float e2[3], k2;
};
// The early-exit walks' own tree: the reference's binary tree with kWideLevels levels collapsed into one node of up to
// kWide children (box_maybe / candidate_reached in ct_traverse.cuh explain why these walks may skip the boxes in between).
// A child is 32 bytes, two 16-byte loads: its box as floats (round to nearest, the same values pairs32 holds) and
// (ref, cnt): cnt > 0 -> leaf holding triangles [ref, ref + cnt); cnt == 0 -> ref = its own wide node.  Children keep the
// reference's DFS order; unused children hold an inverted box (never accepted) and ref = kNoPos.
#ifndef CT_WIDE_LEVELS
#define CT_WIDE_LEVELS 2
#endif
constexpr int kWideLevels = CT_WIDE_LEVELS;
constexpr int kWide = 1 << kWideLevels;
struct __align__(16) DevWideChild { float bmin[3], bmax[3]; uint32_t ref, cnt; };
struct __align__(16) DevWide { DevWideChild c[kWide]; };

struct DevLight { int32_t type; float intensity; double pos[3]; double dir[3]; };
struct DevShadowLight { int32_t type; uint32_t index; double v[3]; };   // non-ambient lights, file order; index = light number
struct __align__(16) OvfRay {        // a parked ray: 64 B
    double o[3], d[3];
    uint32_t target;                 // kAnyHit: word of the occlusion mask; kFirstLine: queue slot of the path
    uint32_t bit;                    // kAnyHit: bit inside that word
};

struct DevSched {                    // zeroed at the start of every tile render
    unsigned long long work[kMaxLaunches];   // dynamic-fetch cursors, one per launch of the tile
    uint32_t queue_count[16];        // paths alive at depth d (d >= 1)
    uint32_t own_count;              // chunks of the tile this device took from the (possibly shared) cursor
    unsigned long long steal_local;  // the cursor of a tile rendered by this device alone
    uint32_t static_next;            // shared frame with a declared partition: next entry of this device's dealt share
    uint32_t ovf_count[40];          // rays parked for the k_overflow launch 2*depth + {0: bounce, 1: shadow}
    uint32_t ovf_cursor[40];         // k_overflow's warp-cooperative pass: next parked ray to take
    uint32_t huge_count[40];         // ... rays it handed on to k_overflow_huge
    uint32_t far_count[16];          // reflection paths of depth d whose shading point may differ from their parent's (far_list)
};
struct DevTotals {                   // running ray / test counters (never reset by a tile)
    unsigned long long rays_primary, rays_shadow, rays_reflection, box_tests, tri_tests;
    unsigned long long rays_overflow;    // rays whose DFS ran past the budget
    unsigned long long rays_in_place;    // ... of which the parking buffer was full: finished by their own thread
    unsigned long long box_exact, tri_exact;   // tests the fp32 filters left to the fp64 arithmetic (CT_FLAG_COUNT_TESTS)
    unsigned long long rays_shadow_reused;     // shadow rays (counted in rays_shadow) that were not traced: an ancestor's identical ray had been
};

struct Params {
    const DevPair32 *pairs32;
    const DevPair64 *pairs64;
    const DevWide *wide;                 // node 0 = the root's children (nullptr: the root is a leaf)
    uint32_t n_wide;
    double root_min[3], root_max[3];     // node 0
    float root_min32[3], root_max32[3];  // ... as floats, for the slab filter
    uint32_t root_ref, root_cnt;
    uint32_t nested;                     // every child's box lies inside its parent's (checked at upload): box_maybe may be used
    double bound[3];                     // >= |b| for every node bound b per axis (+inf disables the filter), see ray_finish
    const DevTri *tris;
    const DevTri32 *tris32;
    const ct_material *materials;    // by original id
    const DevLight *lights;
    const DevShadowLight *slights;
    uint32_t n_lights, n_slights, n_tri, n_nodes, n_pairs;
    uint32_t occ_words;              // words of occlusion bits per path = ceil(n_lights / 32)
    uint32_t pos_of_tri0;            // leaf position of original triangle 0 (closestIndex default, raythread.cpp:205)
    uint32_t budget;                 // see kDefaultBudget
    uint32_t warp_budget;            // see kWarpBudget
    uint32_t any_leaves;             // leaf-list entries an any-hit walk uses (<= kAnyLeaves): 12, or 8 for scenes with 16 or more shadow-casting lights
    uint32_t primary_budget;         // pair visits after which k_primary parks a closest-hit walk for k_primary_long (0: never), see kDefaultPrimaryBudget
    double cam[3], rot[9];
    float vp_w, vp_h, vp_d;
    int W, H, max_depth;
    uint32_t background;
    // tile
    int x_lo, n_x, y_lo, n_y;        // canvas x in [x_lo, x_lo+n_x), n_y traced rows starting at y_lo
    int subsample, n_rows;           // CT_FLAG_SUBSAMPLING: the tile spans n_rows canvas rows of which every other one is traced
    int supersample;                 // CT_FLAG_SUPERSAMPLING: 16 consecutive slots = the 4x4 jittered samples of one pixel
    uint32_t *final_color;           // the traced pixels' / samples' colours by slot, for k_subsample / k_supersample
    int blocks_x;                    // ceil(n_x / 8): pixel blocks of 8x4 per warp
    uint32_t n_slots;                // blocks_x * ceil(n_y/4) * 32
    uint32_t cap;                    // capacity of every per-slot array
    // per-slot path state
    float *hit0_t; uint32_t *hit0_pos;           // depth-0 hit records, by slot (pos = kNoPos: miss)
    float *hitb_t; uint32_t *hitb_pos;           // depth>=1 hits, by queue slot
    double *ray_buf[2];                          // depth>=1 rays: 6 doubles per queue slot, ping-pong
    uint32_t *path_slot[2];                      // queue slot -> depth-0 slot, ping-pong
    uint32_t *parent_q[2];                       // queue slot -> the parent path's queue slot one depth up (kNoReuse bit: its shading point is its own)
    // every depth's arrays, for k_shade's walk up the chain of shading points that coincide (see occlusion_source)
    const uint32_t *parent_q_all; const float *hitb_t_all; const uint32_t *occ_all;
    uint32_t reuse_shadow;                       // option "shadow_reuse"
    uint32_t *far_list;                          // this depth's reflection paths that need shadow rays of their own (k_bounce appends, k_shadow reads)
    uint32_t *occ;                               // [path][occ_words] shadow-ray verdicts of the current depth, bit i = light i occluded
    uint32_t *stack_color; float *stack_refl;    // [depth][slot]
    uint8_t *term_level;                         // [slot] level at which the chain ended
    uint32_t *fb;                                // W*H, this device's framebuffer
    uint32_t *fb_out;                            // where finished pixels are stored: fb, or the root GPU's fb (peer memory)
    unsigned long long *steal;                   // the tile's chunk cursor: local, or on the root GPU (peer memory)
    uint32_t chunk_shift;                        // log2(slots per chunk)
    uint32_t steal_stride;                       // 1; R > 1 (option "emulate_ranks") takes every R-th chunk only: the share of one of R GPUs
    uint32_t part_index, part_count;             // shared frame: this device is participant part_index of part_count (0: not declared)
    uint32_t static_eighths;                     // ... of every 8 * part_count chunks, static_eighths * part_count are dealt, the rest stolen
    uint32_t run_shift;                          // log2 of the run of consecutive chunks that is dealt / stolen as one unit (option "shared_run_shift")
    uint32_t *own_chunks;                        // chunk numbers this device took, in the order it took them
    uint32_t *dbg_found, *dbg_index; float *dbg_t;   // optional (CT_FLAG_KEEP_HITS), framebuffer layout
    // parked rays
    OvfRay *ovf; uint32_t ovf_cap;
    uint32_t *ovf_huge;                          // indices (into ovf) of the rays k_overflow left to k_overflow_huge
    uint32_t *split_path;                        // optional (ct_gpu_debug_primary; NULL in frames): by q, how k_primary_split decided the ray
    const uint32_t *pair_parent;                 // pair -> 2 * parent pair + side of its own box (kNoPos for the root's children pair)
    const uint32_t *tri_parent;                  // leaf position -> 2 * pair + side of the box of the leaf that holds it (kNoPos: root leaf)
    DevSched *sched;
    DevTotals *tot;
    // shade queries (ct_gpu_shade_rays; unused by frames): the caller's rays of the current batch, n_slots x 3 doubles each, read as
    // the depth-0 rays by the QUERY forms of the stage kernels.  Last in the struct: the frame kernels' parameter offsets do not move.
    const double *q_org, *q_dir;
};

struct LocalCount { uint32_t box = 0, tri = 0, box_exact = 0, tri_exact = 0; };

}  // namespace
