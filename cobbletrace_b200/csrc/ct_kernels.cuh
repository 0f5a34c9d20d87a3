// ct_kernels.cuh -- ray generation, work distribution, and the wavefront kernels of one tile
// (k_primary, k_shadow, k_emit, k_shade, k_bounce, k_overflow, k_overflow_huge, k_resolve, k_subsample, k_supersample) plus the KAT kernels.
// Part of the single translation unit ct_gpu.cu (everything lives in its anonymous namespace).
#pragma once

#include "ct_traverse.cuh"

namespace {

// The counter-based stand-in for rand() in the supersampling jitter (the parity harness patches the same
// function into the compiled reference in place of rand(); DESIGN.md, sampling modes).
CT_DEV uint32_t hash3(uint32_t x, uint32_t y, uint32_t k) {
    uint32_t h = x * 0x9E3779B1u ^ (y * 0x85EBCA77u) ^ (k * 0xC2B2AE3Du);
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    return h;
}

// Canvas point of sample k (= 4 xs + ys) of pixel (x, y): the reference's float bookkeeping (raythread.cpp:461-505)
// replayed up to that sample -- sampleX/sampleY are jittered, used, un-jittered and stepped in float, so each
// sample's point depends on the rounding of the ones before it.
CT_DEV void sample_point(int x, int y, int k, float &px, float &py) {
    const float stepsize = 0.25f, jitter = 0.03125f;          // 1/(float)samples, stepsize/8
    float sample_x = (float)x, sample_y = (float)y;
    uint32_t call = 0;
    for (int xs = 0; xs < 4; xs++) {
        sample_y = (float)y;
        for (int ys = 0; ys < 4; ys++) {
            float rx = __fdiv_rn(__int2float_rn((int)(hash3((uint32_t)x, (uint32_t)y, call++) & 0x7fffffffu)), 2147483648.0f);   // (float)RAND_MAX
            float ry = __fdiv_rn(__int2float_rn((int)(hash3((uint32_t)x, (uint32_t)y, call++) & 0x7fffffffu)), 2147483648.0f);
            rx = __fsub_rn(__fmul_rn(rx, 0.0625f), jitter);
            ry = __fsub_rn(__fmul_rn(ry, 0.0625f), jitter);
            sample_x = __fadd_rn(sample_x, rx);
            sample_y = __fadd_rn(sample_y, ry);
            if (xs * 4 + ys == k) { px = sample_x; py = sample_y; return; }
            sample_y = __fadd_rn(__fsub_rn(sample_y, ry), stepsize);
            sample_x = __fsub_rn(sample_x, rx);
        }
        sample_x = __fadd_rn(sample_x, stepsize);
    }
    px = sample_x; py = sample_y;
}

// Primary ray through canvas point (px, py): CanvasToViewport (raythread.cpp:186-194) * camera.rotation (mymath.h:68-75)
CT_DEV Ray primary_ray_at(const Params &P, float px, float py) {
    float hh = (float)P.H;                                  // "Keep it square": both scales use bitmap->height
    double sx = (double)__fdiv_rn(P.vp_w, hh), sy = (double)__fdiv_rn(P.vp_h, hh);
    double vx = __dmul_rn((double)px, sx), vy = __dmul_rn((double)py, sy), vz = (double)P.vp_d;
    Ray r;
    r.o = {P.cam[0], P.cam[1], P.cam[2]};
    r.d.x = __dadd_rn(__dadd_rn(__dmul_rn(vx, P.rot[0]), __dmul_rn(vy, P.rot[3])), __dmul_rn(vz, P.rot[6]));
    r.d.y = __dadd_rn(__dadd_rn(__dmul_rn(vx, P.rot[1]), __dmul_rn(vy, P.rot[4])), __dmul_rn(vz, P.rot[7]));
    r.d.z = __dadd_rn(__dadd_rn(__dmul_rn(vx, P.rot[2]), __dmul_rn(vy, P.rot[5])), __dmul_rn(vz, P.rot[8]));
    r.t = kRayTInit;
    return r;
}

// WHERE A DEPTH-0 RAY COMES FROM AND WHERE ITS COLOUR GOES.  A frame's depth-0 slot is a pixel (or a sample of one) of the tile; a
// shade query's (QUERY, ct_gpu_shade_rays) is the caller's ray `slot` of the current batch.  Only primary_ray, slot_pixel and
// store_pixel know the difference: the stage kernels that call them (k_primary, k_shadow, k_shade, k_resolve) take QUERY as a
// template parameter, everything past depth 0 reads the parking buffers and ray queues and is the same for both.

// Primary ray of depth-0 slot `slot`, whose pixel is (x, y): the pixel centre, or one of its 16 jittered samples.
// QUERY: the caller's ray, ray.t = 1e30f as TraceRay's callers pass it (raythread.cpp:508).
template <bool QUERY = false>
CT_DEV Ray primary_ray(const Params &P, uint32_t slot, int x, int y) {
    if (QUERY) {
        Ray r;
        r.o = ld3(P.q_org + 3ull * slot); r.d = ld3(P.q_dir + 3ull * slot); r.t = kRayTInit;
        return r;
    }
    if (!P.supersample) return primary_ray_at(P, (float)x, (float)y);
    float px, py;
    sample_point(x, y, (int)(slot & 15u), px, py);
    return primary_ray_at(P, px, py);
}

// slot -> canvas pixel.  A warp owns an 8x4 pixel block (coherent rays); returns false for padding lanes
// and for pixels PutPixel would drop (draw2d.h:11-14), which are not traced at all (with subsampling a dropped
// row is still traced -- fb_index = -1 -- because its colour enters the average stored in the row above it).
// QUERY: slot i of the batch is ray i, valid for i < n_slots; fb_index = -1, and store_pixel writes final_color (the caller's colour
// array at the batch's first ray) only.
CT_DEV void store_pixel(const Params &P, uint32_t slot, int fb_index, uint32_t color) {
    if (fb_index >= 0) P.fb_out[fb_index] = color;
    if (P.final_color) P.final_color[slot] = color;
}

template <bool QUERY = false>
CT_DEV bool slot_pixel(const Params &P, uint32_t slot, int &x, int &y, int &fb_index) {
    if (QUERY) { x = y = 0; fb_index = -1; return slot < P.n_slots; }
    if (P.supersample) slot >>= 4;                            // 16 samples per pixel
    uint32_t blk = slot >> 5, lane = slot & 31u;
    int bx = (int)(blk % (uint32_t)P.blocks_x), by = (int)(blk / (uint32_t)P.blocks_x);
    int ix = bx * 8 + (int)(lane & 7u), iy = by * 4 + (int)(lane >> 3);
    if (ix >= P.n_x || iy >= P.n_y) return false;
    x = P.x_lo + ix;
    if (P.subsample)    // raythread.cpp:527-530: y += 2, except that the last row of the partition is always traced
        y = P.y_lo + ((iy == P.n_y - 1 && (P.n_rows & 1) == 0) ? P.n_rows - 1 : 2 * iy);
    else
        y = P.y_lo + iy;
    int col = x + P.W / 2, row = P.H / 2 - y;               // CanvasPutPixel raythread.cpp:181-182
    if (col < 0 || col >= P.W) return false;
    fb_index = row * P.W + col;
    if (row < 0 || row >= P.H) {
        if (!P.subsample) return false;
        fb_index = -1;                                       // traced for the average of the row above it, never stored
    }
    if (P.supersample) fb_index = -1;                        // a sample: k_supersample blends the 16 of a pixel and stores it
    return true;
}

CT_DEV unsigned long long warp_fetch(unsigned long long *cursor) {   // persistent warps pull 32 work items at a time
    unsigned long long base = 0;
    if ((threadIdx.x & 31u) == 0) base = atomicAdd(cursor, 32ull);
    return __shfl_sync(0xffffffffu, base, 0);
}

CT_DEV void warp_add(unsigned long long *dst, uint32_t v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31u) == 0 && v) atomicAdd(dst, (unsigned long long)v);
}

// Depth-0 paths are numbered in the order this device took their chunks from the cursor.
CT_DEV uint32_t own_slot(const Params &P, uint32_t q) {
    return (P.own_chunks[q >> P.chunk_shift] << P.chunk_shift) + (q & ((1u << P.chunk_shift) - 1u));
}
CT_DEV uint32_t depth0_count(const Params &P) { return P.sched->own_count << P.chunk_shift; }

// The path with queue index q at `depth`: its ray (direction only for depth 0 is regenerated from the pixel),
// its closest-hit record and its depth-0 slot.  False for padding lanes / untraced pixels.
template <bool QUERY = false>
CT_DEV bool load_path(const Params &P, int depth, uint32_t q, uint32_t &slot, int &fbi, Ray &r, float &tc, uint32_t &pos) {
    if (depth == 0) {
        int x, y;
        slot = own_slot(P, q);
        if (!slot_pixel<QUERY>(P, slot, x, y, fbi)) return false;
        tc = P.hit0_t[slot]; pos = P.hit0_pos[slot];
        if (pos == kNoPos) return true;                         // a miss: nobody needs its ray again (background pixel)
        r = primary_ray<QUERY>(P, slot, x, y);
    } else {
        const int cur = depth & 1;
        slot = P.path_slot[cur][q];
        fbi = 0;
        const double2 *rb = reinterpret_cast<const double2 *>(P.ray_buf[cur] + 6ull * q);
        double2 a = rb[0], b = rb[1], c = rb[2];
        r.o = {a.x, a.y, b.x}; r.d = {b.y, c.x, c.y}; r.t = 0.0f;
        tc = P.hitb_t[q]; pos = P.hitb_pos[q];
        if (pos == kNoPos) pos = P.pos_of_tri0;                 // "closestIndex = 0" (raythread.cpp:205): no barycentric pass at all
    }
    return true;
}

// IDENTICAL SHADOW RAYS ARE TRACED ONCE.  The reference's reflection rays are built with t = 0 (raythread.cpp:373, SURVEY 0.4): a
// reflection "hit" -- the first triangle in DFS order whose line passes -- has tclosest = 0, so the next shading point is
// position = origin + 0 * direction = the ray's origin = the PREVIOUS shading point, bit for bit (raythread.cpp:360; the direction
// must be finite for 0 * direction to be 0).  ComputeLighting then casts, for every light, exactly the shadow ray the previous
// level already cast from that point (raythread.cpp:288-304: same origin, same light, t = 1e30f): same ray, same verdict
// (k_emit checks the "bit for bit" when it builds the reflection ray and flags the exceptions: kNoReuse).  So
// a path whose hit has tclosest == 0 takes its occlusion mask from its parent (and so on up the chain) instead of tracing
// the rays again; only normal, material and view direction differ between the levels.  The rays still count as shadow rays
// (rays_shadow keeps the reference's definition); rays_shadow_reused says how many of them were answered this way.
// Is the shading point of path q at `depth` (>= 1) a copy of its parent's?
CT_DEV bool shading_point_repeats(const Params &P, int depth, uint32_t q) {
    if (!P.reuse_shadow || depth <= 0) return false;
    const size_t i = (size_t)depth * P.cap + q;
    return __ldg(P.hitb_t_all + i) == 0.0f && !(__ldg(P.parent_q_all + i) & kNoReuse);
}
// The occlusion mask path q of `depth` is lit with: its own, or that of the nearest ancestor whose shading point it repeats.
CT_DEV const uint32_t *occlusion_source(const Params &P, int depth, uint32_t q) {
    while (shading_point_repeats(P, depth, q)) { q = __ldg(P.parent_q_all + (size_t)depth * P.cap + q) & ~kNoReuse; depth--; }
    return P.occ_all + ((size_t)depth * P.cap + q) * P.occ_words;
}

CT_DEV void clear_occ(const Params &P, uint32_t q) {
    for (uint32_t w = 0; w < P.occ_words; w++) P.occ[(size_t)q * P.occ_words + w] = 0u;
}

// Park a ray for k_overflow.  False when the buffer is full (the caller then finishes the ray in place).
CT_DEV bool park_ray(const Params &P, int ovf_idx, const double *r64, uint32_t target, uint32_t bit) {
    uint32_t i = atomicAdd(&P.sched->ovf_count[ovf_idx], 1u);
    if (i >= P.ovf_cap) { atomicAdd(&P.tot->rays_in_place, 1ull); return false; }
    OvfRay &o = P.ovf[i];
    o.o[0] = r64[0]; o.o[1] = r64[1]; o.o[2] = r64[2];
    o.d[0] = r64[3]; o.d[1] = r64[4]; o.d[2] = r64[5];
    o.target = target; o.bit = bit;
    return true;
}

// The per-ray loop of the early-exit kernels (k_shadow, k_bounce, k_debug_early): the walk with the budget; a walk given up at the
// budget is parked for k_overflow (target / bit: where k_overflow stores the answer), or -- parking buffer full -- walked again
// right here without a budget.  A shadow ray whose origin lies so far outside the scene that every box passes (a shading point 2^32
// ray lengths away, SURVEY 0.4) is parked at its first visit: no point in walking up to the budget first, k_overflow hands it
// straight to k_overflow_huge.  WARP-LEVEL: every lane calls it.  Returns, for an active lane, how the ray was finished (kWalked,
// kParked, kInPlace); finish(res, tc, pos) receives the answer of a walk that was not given up, over(parked) hears of one that was.
enum { kWalked = 0, kParked = 1, kInPlace = 3 };
template <TraverseMode MODE, bool COUNT, class Finish, class Over>
CT_DEV int walk_or_park(const Params &P, const TRay &r, const double *r64, bool active, uint32_t budget, int ovf_idx, uint32_t target,
                        uint32_t bit, uint32_t &n_parked, LocalCount &lc, uint32_t *sm, Finish &&finish, Over &&over) {
    if (MODE == kAnyHit && active && (double)r.om > 0x1p20 * fmax(fmax(P.bound[0], P.bound[1]), P.bound[2])) budget = 0u;
    int how = kWalked;
    while (true) {                                                      // warp-uniform: traverse_early is warp-synchronous
        float tc; uint32_t pos;
        const int res = traverse_early_any<MODE, COUNT>(P, r, active, budget, tc, pos, lc, sm);
        bool again = false;
        if (active) {
            if (res == kTravOverBudget) {
                n_parked++;
                again = !park_ray(P, ovf_idx, r64, target, bit);        // parking buffer full: finish in place, no budget
                budget = 0xffffffffu;
                how = again ? kInPlace : kParked;
                over(!again);
            } else {
                finish(res, tc, pos);
            }
        }
        active = again;
        if (!__any_sync(kFullMask, again)) break;
    }
    return how;
}

// Primary rays.  Persistent warps take chunks of 32 or 64 slots from the tile's cursor -- one counter for the whole
// tile, which in a multi-GPU frame lives on the root GPU and is shared by all devices over NVLink (dynamic
// stealing at chunk granularity, SURVEY 8e) -- and remember which chunks they took: the later stages of this
// device work on exactly those.
// Which chunk of the tile does this warp trace next?  (called by lane 0)
//   one device, or a shared frame without a declared partition: the next one from the cursor (P.steal: this device's own
//     or, shared, the root GPU's over NVLink) -- pure dynamic stealing;
//   shared frame of R declared participants: the chunks are numbered in groups of 8R; of every group the first E*R are
//     DEALT (participant r owns r, r + R, ...: no atomics on another GPU, and -- being interleaved at 32-pixel grain --
//     an equal share of every later stage's work too), the other (8 - E)*R are STOLEN from the root's cursor (absorbs a
//     slower or busier GPU).  Stealing everything balances only this kernel: the GPU that holds the cursor steals
//     cheaper and ends up with more paths to light (measured at 8 GPUs: 1.75 ms on the root against 1.41 ms elsewhere).
CT_DEV bool next_chunk(const Params &P, uint32_t n_chunks, bool &dealt_left, uint32_t &idx) {
    // Chunks are handed out in RUNS of L = 2^run_shift consecutive chunks (horizontally adjacent 8x4 blocks): the formulas
    // below deal / steal run numbers, `off` walks through a run.  L = 1 is the finest interleave; a longer run keeps the warps
    // of one GPU on neighbouring pixels (option "shared_run_shift").
    const uint32_t R = P.part_count, E = P.static_eighths, rs = P.run_shift, L = 1u << rs;
    if (R <= 1u) {
        if (P.steal_stride <= 1u) {
            const unsigned long long d = atomicAdd(P.steal, 1ull);
            idx = (uint32_t)d;
            return d < n_chunks;
        }
        while (true) {                                       // (option "emulate_ranks": the runs rank 0 of steal_stride GPUs would own)
            const unsigned long long c = atomicAdd(P.steal, 1ull);
            const unsigned long long run = (c >> rs) * P.steal_stride;
            if ((run << rs) >= n_chunks) return false;
            idx = (uint32_t)((run << rs) + (c & (L - 1u)));
            if (idx < n_chunks) return true;
        }
    }
    const uint32_t n_runs = (n_chunks + L - 1u) >> rs;
    const uint32_t G = 8u * R, n_groups = (n_runs + G - 1u) / G;
    while (dealt_left) {
        const uint32_t c = atomicAdd(&P.sched->static_next, 1u);
        const uint32_t cr = c >> rs, off = c & (L - 1u);
        const uint32_t g = cr / E;
        if (g >= n_groups) { dealt_left = false; break; }
        idx = ((g * G + (cr - g * E) * R + P.part_index) << rs) + off;
        if (idx < n_chunks) return true;
    }
    const uint32_t per = (8u - E) * R;
    while (per) {
        const unsigned long long d = atomicAdd(P.steal, 1ull);
        const unsigned long long dr = d >> rs, off = d & (L - 1u);
        const unsigned long long g = dr / per;
        if (g >= n_groups) break;
        idx = (uint32_t)(((g * G + E * R + (dr - g * per)) << rs) + off);
        if (idx < n_chunks) return true;
    }
    return false;
}

CT_DEV void emit_paths(const Params &P, int depth, bool active, uint32_t q, uint32_t slot, V3 o, V3 d, float tc, uint32_t pos, uint32_t &n_refl);

// The closest-hit record of the depth-0 path (slot, q): ClosestIntersection's results as TraceRay sees them (raythread.cpp:227, :205).
CT_DEV void store_primary_hit(const Params &P, uint32_t slot, uint32_t q, int fbi, bool found, float tc, uint32_t pos) {
    CT_CHECK(slot < P.cap && q < P.cap);
    P.hit0_t[slot] = tc;
    P.hit0_pos[slot] = found ? (pos == kNoPos ? P.pos_of_tri0 : pos) : kNoPos;
    if (found) clear_occ(P, q);
    if (P.dbg_found && fbi >= 0) {
        P.dbg_found[fbi] = found ? 1u : 0u;
        P.dbg_index[fbi] = (pos == kNoPos) ? 0u : P.tris[pos].orig;
        P.dbg_t[fbi] = tc;
    }
}

// k_primary's rays: the warp takes chunks from the tile's cursor (next_chunk) and hands the slots of its current chunk to
// its lanes, 32 at a time.
struct PrimaryJob {
    uint32_t n_chunks, chunk;
    bool dealt_left;                                        // lane 0's view of this device's dealt share
    uint32_t pend_slot = 0, pend_q = 0, pend_left = 0;      // warp-uniform: what is left of the chunk being handed out
    uint32_t slot = 0, q = 0; int fbi = -1;                 // this lane's ray
    uint32_t n_rays = 0;

    // One slot per lane (got: the slot is a pixel to trace, r / r64 set up); false once the cursor is exhausted.
    template <bool QUERY>
    CT_DEV bool refill(const Params &P, bool &got, TRay &r, double *r64) {
        const uint32_t lane = threadIdx.x & 31u;
        if (pend_left == 0u) {
            unsigned long long base = ~0ull;
            uint32_t mine = 0;
            if (lane == 0) {
                uint32_t idx;
                if (next_chunk(P, n_chunks, dealt_left, idx)) {
                    base = (unsigned long long)idx << P.chunk_shift;
                    mine = atomicAdd(&P.sched->own_count, 1u);
                    CT_CHECK(mine <= (P.cap >> kChunkLocalShift));
                    P.own_chunks[mine] = idx;
                }
            }
            base = __shfl_sync(kFullMask, base, 0);
            mine = __shfl_sync(kFullMask, mine, 0);
            if (base == ~0ull) return false;
            pend_slot = (uint32_t)base; pend_q = mine << P.chunk_shift; pend_left = chunk;
        }
        // rank == lane, written as the popcount of the lanes below it: with the plain `lane` k_primary compiles to other SASS
        // (more spills), which measured slower together with traverse_closest's plain push (see there)
        const uint32_t take = min(32u, pend_left), rank = __popc((1u << lane) - 1u);
        if (rank < take) {
            slot = pend_slot + rank; q = pend_q + rank;     // q: this path's depth-0 number on this device
            int x, y;
            if (slot < P.n_slots && slot_pixel<QUERY>(P, slot, x, y, fbi)) {
                const Ray ray = primary_ray<QUERY>(P, slot, x, y);
                tray_setup(r, ray, P.bound, r64);
                got = true;
            }
        }
        pend_slot += take; pend_q += take; pend_left -= take;
        return true;
    }
    CT_DEV void finish(const Params &P, bool found, float tc, uint32_t pos) {
        n_rays++;
        store_primary_hit(P, slot, q, fbi, found, tc, pos);
    }
};

// The per-ray loop of the primary rays (k_primary, k_debug_primary): the closest-hit walk (ray.t = 1e30f), under PARK with a budget
// of P.primary_budget pair visits when parking buffers exist.  A walk given up at the budget is parked for k_primary_long /
// k_primary_split (target / bit: the path's q and slot), or -- parking buffer full -- walked again right here without a budget,
// from ray.t = 1e30f: the walk given up has already lowered r.t.  WARP-LEVEL: every lane calls it.  Returns, for a lane with a ray,
// how it was finished (kWalked, kParked, kInPlace); res / tc / pos are the answer of a ray that was not parked.
template <bool COUNT, bool PARK>
CT_DEV int primary_walk_or_park(const Params &P, TRay &r, const double *r64, bool got, uint32_t target, uint32_t bit, uint32_t &n_parked,
                                LocalCount &lc, int &res, float &tc, uint32_t &pos) {
    const uint32_t budget = (PARK && P.primary_budget > 0u && P.ovf != nullptr) ? P.primary_budget : 0xffffffffu;
    res = traverse_closest<COUNT, PARK>(P, r, got, tc, pos, lc, nullptr, budget);   // warp-synchronous
    int how = kWalked;
    const bool over = PARK && got && res == kTravOverBudget;
    if (PARK && __any_sync(kFullMask, over)) {
        bool redo = false;
        if (over) { const bool parked = park_ray(P, 0, r64, target, bit); redo = !parked; how = parked ? kParked : kInPlace; n_parked++; }
        if (__any_sync(kFullMask, redo)) {
            if (redo) r.t = kRayTInit;
            float tc2; uint32_t pos2;
            const int res2 = traverse_closest<COUNT>(P, r, redo, tc2, pos2, lc);
            if (redo) { res = res2; tc = tc2; pos = pos2; }
        }
    }
    return how;
}

// Primary rays.  Persistent warps take chunks of 32 (or 64) slots from the tile's cursor (next_chunk) and remember which
// chunks they took: the later stages of this device work on exactly those.  A warp walks 32 rays of a chunk together (one
// 8x4 pixel block: neighbouring rays visit the same nodes; refilling idle lanes from the next chunk instead measured slower,
// DESIGN.md 5).
// PARK: walks longer than P.primary_budget pair visits are given up and parked for k_primary_long (option "primary_budget").
// QUERY: the depth-0 rays are a shade query's (see primary_ray).
template <bool COUNT, bool PARK, bool QUERY = false>
__global__ void __launch_bounds__(kBlockThreads, kMinBlocks) k_primary(const __grid_constant__ Params P) {
    LocalCount lc;
    uint32_t n_refl = 0;
    PrimaryJob job;
    job.chunk = 1u << P.chunk_shift;
    job.n_chunks = (P.n_slots + job.chunk - 1u) >> P.chunk_shift;
    job.dealt_left = P.part_count > 1u && P.static_eighths > 0u;
    uint32_t n_parked = 0;
    while (true) {
        bool got = false;
        double r64[kRay64];
        TRay r;
        if (!job.refill<QUERY>(P, got, r, r64)) break;
        int res; float tc; uint32_t pos;
        const int how = primary_walk_or_park<COUNT, PARK>(P, r, r64, got, job.q, job.slot, n_parked, lc, res, tc, pos);
        const bool done = got && how != kParked, found = res == kTravHit;
        if (done) job.finish(P, found, tc, pos);
        if (P.max_depth > 0)          // the recursion step at once, while ray and hit are at hand (no k_emit pass over the tile)
            emit_paths(P, 0, done, job.q, job.slot, {r64[0], r64[1], r64[2]}, {r64[3], r64[4], r64[5]}, tc,
                       found ? (pos == kNoPos ? P.pos_of_tri0 : pos) : kNoPos, n_refl);
    }
    warp_add(&P.tot->rays_reflection, n_refl);
    warp_add(&P.tot->rays_primary, job.n_rays);
    warp_add(&P.tot->rays_overflow, n_parked);
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// The primary rays k_primary parked (walks longer than P.primary_budget pair visits), 32 to a warp: the same closest-hit walk from
// the start, without a budget, then the hit record and the recursion step exactly as k_primary does them.  A long walk in
// k_primary has the other 31 lanes of its 8x4 block waiting; here its neighbours are long walks too.
template <bool COUNT>
__global__ void __launch_bounds__(kBlockThreads, kMinBlocks) k_primary_long(const __grid_constant__ Params P, int work_idx) {
    const uint32_t n = min(P.sched->ovf_count[0], P.ovf_cap);
    if (n == 0) return;
    LocalCount lc;
    uint32_t n_refl = 0, n_rays = 0;
    while (true) {
        const unsigned long long base = warp_fetch(&P.sched->work[work_idx]);
        if (base >= n) break;
        const uint32_t i = (uint32_t)base + (threadIdx.x & 31u);
        const bool active = i < n;
        double r64[kRay64];
        TRay r;
        uint32_t q = 0, slot = 0;
        if (active) {
            const OvfRay &o = P.ovf[i];
            Ray ray; ray.o = ld3(o.o); ray.d = ld3(o.d); ray.t = kRayTInit;
            q = o.target; slot = o.bit;
            tray_setup(r, ray, P.bound, r64);
        }
        float tc; uint32_t pos;
        const bool found = traverse_closest<COUNT>(P, r, active, tc, pos, lc) == kTravHit;
        if (active) {
            // (the pixel only for CT_FLAG_KEEP_HITS: a shade query's parked rays get a meaningless fbi here, which
            // store_primary_hit ignores because a query's dbg_* are NULL -- so this kernel needs no QUERY form)
            int x, y, fbi = -1;
            if (!slot_pixel(P, slot, x, y, fbi)) fbi = -1;
            n_rays++;
            store_primary_hit(P, slot, q, fbi, found, tc, pos);
        }
        if (P.max_depth > 0)
            emit_paths(P, 0, active, q, slot, {r64[0], r64[1], r64[2]}, {r64[3], r64[4], r64[5]}, tc,
                       found ? (pos == kNoPos ? P.pos_of_tri0 : pos) : kNoPos, n_refl);
    }
    warp_add(&P.tot->rays_reflection, n_refl);
    warp_add(&P.tot->rays_primary, n_rays);
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// IntersectBVHClosest as an ORDER-FREE search (primary rays, ray.t = 1e30f).  On a nested tree the reference tests a triangle
// iff its LEAF's own box passes IntersectAABB against the ray.t of that moment (DESIGN.md 2: ray.t only ever decreases, so
// tmin(ancestor) <= tmin(leaf) < ray.t at the leaf's visit <= ray.t at the ancestor's visit).  Let G be the triangles with a
// barycentric pass and 1e-4 < t < 1e30 whose leaf box passes the two conditions that do not involve ray.t, m = min t over G,
// and sigma the ray's slop bound (tray_nearest_setup:  tmin(leaf of Z) <= t_Z + sigma  for every Z).  Then
//   * ray.t never drops below m; the first triangle with t = m is tested unless ray.t <= tmin(its leaf) <= m + sigma by
//     then -- either way the walk ends with ray.t <= m + sigma;
//   * a triangle with t > tau changes the fate of one with t <= tau only by lowering ray.t to a value that blocks the
//     latter's leaf, i.e. only if  tmin(that leaf) >= t > tau.
// So with S = { Z in G : t_Z <= m + sigma }:  if every member of S has tmin(leaf) <= m + sigma, nothing outside S can block
// a member of S, a tested member of S lowers ray.t below anything outside S, and replaying the reference's update rules
// (bvh.cpp:161, 178, 212) over S alone, in leaf-position order (= the reference's test order), gives the reference's
// ray.t, tclosest and closestIndex bit for bit.  Finding S needs no particular order: the search keeps best = min t so far
// and prunes a box only when the LOWER end of its near bracket is >= best + 2 sigma: every triangle Z below it has
// t_Z >= tmin(leaf of Z) - sigma >= tmin(box) - sigma >= best + sigma >= m + sigma (boxes are nested, best >= m; sigma
// carries slack, so the inequality is strict) and is not in S.  Each barycentric pass within best + sigma becomes a
// candidate once the exact fp64 test of its own leaf box confirms membership in G (that test also yields the reference's
// tmin for the replay).  The argument is checked on the CPU by tests/test_free_closest_prototype.py.
//
// The parked primary rays, ONE RAY PER WARP (option "primary_split"): that search run as a frontier.  Per round every lane
// takes one pending node of the wide tree off a stack the warp shares, tests its four children conservatively against
// best + 2 sigma, tests accepted leaves on the spot (a barycentric pass within best + sigma becomes a candidate) and hands
// accepted interior children back; the warp-wide minimum of t is exchanged once per round.  Afterwards the lanes' candidates
// within sigma of the minimum (S) are gathered and lane 0 replays the reference's update rules over them in leaf order (= the
// reference's test order where leaf positions increase along the DFS; render_impl sends the parked rays of other trees to
// k_primary_long) -- the CPU prototype tests/test_free_closest_prototype.py::test_frontier_walk_equals_reference_walk.
// A walk of ~300 DEPENDENT pair visits (the floor under k_primary, DESIGN.md 6) becomes ~12 rounds: a round descends two levels of
// the reference's tree whatever the number of boxes the ray grazes.  Undecided rays (more than kNearCand candidates in a lane or 32
// in the warp, a candidate whose leaf starts beyond the minimum + sigma, t >= FINF, a full stack, rays outside the slop analysis)
// are walked by lane 0 in the reference's order.  P.split_path (ct_gpu_debug_primary only) receives 2 | outcome << 8 by q,
// outcome one of kSplit*.
constexpr int kNearCand = 4;             // candidates per lane
constexpr int kSplitStack = 512;         // pending wide nodes per warp: (node, lower end of its near bracket)
enum { kSplitDecided = 0, kSplitNoSigma = 1, kSplitNotNested = 2, kSplitFinf = 3, kSplitCandFull = 4, kSplitStackFull = 5,
       kSplitLate = 6, kSplitMany = 7 };
template <bool COUNT>
__global__ void __launch_bounds__(kOvfThreads) k_primary_split(const __grid_constant__ Params P) {
    const uint32_t n = min(P.sched->ovf_count[0], P.ovf_cap);
    if (n == 0) return;
    LocalCount lc;
    uint32_t n_refl = 0, n_rays = 0;
    const uint32_t lane = threadIdx.x & 31u;
    __shared__ uint32_t wnode[kOvfThreads / 32][kSplitStack];
    __shared__ float wnear[kOvfThreads / 32][kSplitStack];
    uint32_t *const stk = wnode[threadIdx.x >> 5];
    float *const stk_near = wnear[threadIdx.x >> 5];
    while (true) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&P.sched->ovf_cursor[0], 1u);
        idx = __shfl_sync(kFullMask, idx, 0);
        if (idx >= n) break;
        const OvfRay &o = P.ovf[idx];
        Ray ray; ray.o = ld3(o.o); ray.d = ld3(o.d); ray.t = kRayTInit;
        const uint32_t q = o.target, slot = o.bit;
        double r64[kRay64];
        TRay r;
        tray_setup(r, ray, P.bound, r64);                 // every lane holds the same ray
        tray_nearest_setup(r, P.bound);
        bool ordered = !(r.sg > 0.0f) || P.nested == 0u || P.wide == nullptr;      // warp-uniform: lane 0 walks in the reference's order
        bool found = false;
        float tc = kFinf;                                 // raythread.cpp:204
        uint32_t pos = kNoPos;
        uint32_t why = kSplitDecided;                     // why an ordered walk decides the ray (kSplit*), for P.split_path
        if (!ordered) {
            if (COUNT && lane == 0) lc.box++;
            if (root_accept(P, r)) {
                float cand_t[kNearCand], cand_tmin[kNearCand];
                uint32_t cand_pos[kNearCand], cand_code[kNearCand];
                int ncand = 0;
                uint32_t undecided = 0;                                            // bit 0: a t >= FINF, bit 1: a full candidate list
                float best = kRayTInit, band = kRayTInit, thr = kRayTInit;          // this lane's view; made warp-wide once per round
                if (lane == 0) { stk[0] = 0u; stk_near[0] = -kRayTInit; }
                __syncwarp();
                uint32_t sp = 1;
                while (sp > 0) {
                    const uint32_t take = min(sp, 32u);
                    sp -= take;
                    uint32_t n_out = 0, out_ref[kWide];
                    float out_near[kWide];
                    if (lane < take && stk_near[sp + lane] < thr) {
                        const float4 *qn = reinterpret_cast<const float4 *>(P.wide + stk[sp + lane]);
                        if (COUNT) lc.box += kWide;
#pragma unroll
                        for (int e = 0; e < kWide; e++) {
                            float4 a; uint4 b;
                            ldg256(qn + 2 * e, a, b);
                            const float bmax1 = __uint_as_float(b.x), bmax2 = __uint_as_float(b.y);
                            const bool px = r.rdf[0] > 0.0f, py = r.rdf[1] > 0.0f, pz = r.rdf[2] > 0.0f;
                            const float n0 = __fmaf_rd(px ? a.x : a.w, r.rdf[0], r.cl[0]), f0 = __fmaf_ru(px ? a.w : a.x, r.rdf[0], r.cu[0]);
                            const float n1 = __fmaf_rd(py ? a.y : bmax1, r.rdf[1], r.cl[1]), f1 = __fmaf_ru(py ? bmax1 : a.y, r.rdf[1], r.cu[1]);
                            const float n2 = __fmaf_rd(pz ? a.z : bmax2, r.rdf[2], r.cl[2]), f2 = __fmaf_ru(pz ? bmax2 : a.z, r.rdf[2], r.cu[2]);
                            const float near_lo = fmaxf(fmaxf(n0, n1), n2), far_hi = fminf(fminf(f0, f1), f2);      // box_maybe's brackets
                            if ((far_hi < near_lo) | (far_hi <= 0.0f) | (near_lo >= thr)) continue;
                            if (b.w == 0u) { out_ref[n_out] = b.z; out_near[n_out] = near_lo; n_out++; continue; }
                            for (uint32_t k = 0; k < b.w; k++) {                       // a leaf: its triangles on the spot
                                const uint32_t tp = b.z + k;
                                if (COUNT) lc.tri++;
                                const TriHit th = leaf_triangle<false, COUNT>(P, r, tp, lc);
                                if (!(th.hit & (th.t > kEps) & (th.t < kRayTInit))) continue;      // would not lower a ray.t of 1e30f (bvh.cpp:161)
                                if (!(th.t < kFinf)) { undecided |= 1u; continue; }
                                if (!(th.t <= band)) continue;
                                const uint32_t code = __ldg(P.tri_parent + tp);        // the triangle's leaf: 2 * pair + side
                                if (COUNT) lc.box_exact++;
                                const BoxTimes bt = code == kNoPos ? box_times(r.r64, P.root_min, P.root_max) : exact_child(P.pairs64, code >> 1, code & 1u, r.r64);
                                if (!((bt.tmax >= bt.tmin) & (bt.tmax > 0.0f))) continue;          // a leaf the reference cannot reach
                                if (th.t < best) { best = th.t; band = __fadd_ru(best, r.sg); thr = __fadd_ru(band, r.sg); }
                                if (ncand == kNearCand) {                              // drop what has fallen out of the band
                                    int m = 0;
                                    for (int j = 0; j < kNearCand; j++)
                                        if (cand_t[j] <= band) { cand_t[m] = cand_t[j]; cand_tmin[m] = cand_tmin[j]; cand_pos[m] = cand_pos[j]; cand_code[m] = cand_code[j]; m++; }
                                    ncand = m;
                                }
                                if (ncand == kNearCand) undecided |= 2u;
                                else { cand_t[ncand] = th.t; cand_tmin[ncand] = bt.tmin; cand_pos[ncand] = tp; cand_code[ncand] = code; ncand++; }
                            }
                        }
                    }
                    __syncwarp();                                     // every lane has read its entry before the pushes below
                    // the round's exchange: the minimum of t, "some lane cannot decide", where the accepted children go
                    float bw = best;
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) bw = fminf(bw, __shfl_xor_sync(kFullMask, bw, d));
                    if (bw < best) { best = bw; band = __fadd_ru(best, r.sg); thr = __fadd_ru(band, r.sg); }
                    uint32_t incl = n_out;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(kFullMask, incl, d); if ((int)lane >= d) incl += v; }
                    const uint32_t total = __shfl_sync(kFullMask, incl, 31);
                    if (__any_sync(kFullMask, undecided) || sp + total > (uint32_t)kSplitStack) {
                        const uint32_t u = __reduce_or_sync(kFullMask, undecided);
                        why = (u & 1u) ? kSplitFinf : (u & 2u) ? kSplitCandFull : kSplitStackFull;
                        ordered = true;
                        break;
                    }
                    const uint32_t at = sp + incl - n_out;
                    for (uint32_t k = 0; k < n_out; k++) { stk[at + k] = out_ref[k]; stk_near[at + k] = out_near[k]; }
                    sp += total;
                    __syncwarp();
                }
                if (!ordered && best != kRayTInit) {
                    // ---- S = the candidates within sigma of the minimum, gathered into the (now empty) stack, replayed by lane 0
                    int m = 0;
                    bool late = false;                                // a member of S whose leaf starts beyond the minimum + sigma
                    for (int j = 0; j < ncand; j++)
                        if (cand_t[j] <= band) {
                            late |= !(cand_tmin[j] <= band);
                            cand_t[m] = cand_t[j]; cand_tmin[m] = cand_tmin[j]; cand_pos[m] = cand_pos[j]; cand_code[m] = cand_code[j]; m++;
                        }
                    uint32_t incl = (uint32_t)m;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { const uint32_t v = __shfl_up_sync(kFullMask, incl, d); if ((int)lane >= d) incl += v; }
                    const uint32_t total = __shfl_sync(kFullMask, incl, 31);
                    if (__any_sync(kFullMask, late) || total > 32u) { why = __any_sync(kFullMask, late) ? kSplitLate : kSplitMany; ordered = true; }
                    else {
                        uint32_t *const g_pos = stk, *const g_code = stk + 32;
                        float *const g_t = stk_near, *const g_tmin = stk_near + 32;
                        const uint32_t at = incl - (uint32_t)m;
                        for (int j = 0; j < m; j++) { g_t[at + j] = cand_t[j]; g_tmin[at + j] = cand_tmin[j]; g_pos[at + j] = cand_pos[j]; g_code[at + j] = cand_code[j]; }
                        __syncwarp();
                        if (lane == 0) {
                            for (uint32_t j = 1; j < total; j++) {                    // leaf-position order = the reference's test order
                                const float zt = g_t[j], zm = g_tmin[j]; const uint32_t zp = g_pos[j], zc = g_code[j];
                                uint32_t k = j;
                                while (k > 0 && g_pos[k - 1] > zp) { g_t[k] = g_t[k - 1]; g_tmin[k] = g_tmin[k - 1]; g_pos[k] = g_pos[k - 1]; g_code[k] = g_code[k - 1]; k--; }
                                g_t[k] = zt; g_tmin[k] = zm; g_pos[k] = zp; g_code[k] = zc;
                            }
                            float rt = kRayTInit;
                            uint32_t entered = 0xfffffffeu;                               // (no leaf has this code)
                            for (uint32_t j = 0; j < total; j++) {
                                if (g_code[j] != entered) {                                // the box is tested once per leaf visit
                                    if (!(g_tmin[j] < rt)) continue;                       // bvh.cpp:178, the leaf's own box
                                    entered = g_code[j];
                                }
                                rt = macro_min(rt, g_t[j]);                                // bvh.cpp:161
                                if (rt != kRayTInit && rt < tc) { pos = g_pos[j]; tc = rt; }   // bvh.cpp:212
                            }
                            found = rt != kRayTInit;
                        }
                        __syncwarp();
                    }
                }
            }
        }
        if (ordered) {                                        // warp-uniform
            float tc2; uint32_t pos2;
            const int res = traverse_closest<COUNT>(P, r, lane == 0, tc2, pos2, lc);
            found = res == kTravHit; tc = tc2; pos = pos2;
        }
        if (lane == 0) {                                      // lane 0 holds the answer
            int x, y, fbi = -1;                               // (for CT_FLAG_KEEP_HITS only; a shade query's: see k_primary_long)
            if (!slot_pixel(P, slot, x, y, fbi)) fbi = -1;
            n_rays++;
            store_primary_hit(P, slot, q, fbi, found, tc, pos);
            if (P.split_path) {
                if (ordered && why == kSplitDecided) why = !(r.sg > 0.0f) ? kSplitNoSigma : kSplitNotNested;     // ordered from the start
                P.split_path[q] = 2u | (why << 8);
            }
        }
        if (P.max_depth > 0)
            emit_paths(P, 0, lane == 0, q, slot, {r64[0], r64[1], r64[2]}, {r64[3], r64[4], r64[5]}, tc,
                       found ? (pos == kNoPos ? P.pos_of_tri0 : pos) : kNoPos, n_refl);
        __syncwarp();
    }
    warp_add(&P.tot->rays_reflection, n_refl);
    warp_add(&P.tot->rays_primary, n_rays);
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// ComputeLighting's shadow rays (raythread.cpp:288-306) for the paths alive at `depth`.  Work item =
// (shadow light j, path q), j-major, so the 32 lanes of a warp trace 32 neighbouring shading points towards
// the same light.  Verdicts go to the per-path occlusion mask read by k_shade.
#ifndef CT_SHADOW_BLOCKS
#define CT_SHADOW_BLOCKS CT_MIN_BLOCKS
#endif
template <bool COUNT, bool QUERY = false>
__global__ void __launch_bounds__(kBlockThreads, CT_SHADOW_BLOCKS) k_shadow(const __grid_constant__ Params P, int depth, int work_idx, int ovf_idx) {
    LocalCount lc;
    uint32_t n_shadow = 0, n_parked = 0, n_reused = 0;
    __shared__ uint32_t walk_sm[kWalkWords * kBlockThreads];          // the any-hit walk's per-lane stack and leaf list (traverse_wide)
    uint32_t *const sm = walk_sm + threadIdx.x;
    // depth >= 1 with shadow reuse: only the paths of the far list cast rays of their own; the others are counted here
    const bool use_far = depth > 0 && P.reuse_shadow != 0u;
    const uint32_t n_paths = depth == 0 ? depth0_count(P) : P.sched->queue_count[depth];
    const uint32_t n = use_far ? P.sched->far_count[depth] : n_paths;
    if (use_far && blockIdx.x == 0 && threadIdx.x == 0) {
        const unsigned long long rest = (unsigned long long)(n_paths - n) * P.n_slights;
        atomicAdd(&P.tot->rays_shadow, rest); atomicAdd(&P.tot->rays_shadow_reused, rest);
    }
    const unsigned long long n_pad = ((unsigned long long)n + 31ull) & ~31ull;
    const unsigned long long total = n_pad * P.n_slights;
    while (true) {
        unsigned long long base = warp_fetch(&P.sched->work[work_idx]);
        if (base >= total) break;
        uint32_t j = (uint32_t)(base / n_pad);
        uint32_t q = (uint32_t)(base - (unsigned long long)j * n_pad) + (threadIdx.x & 31u);
        uint32_t slot, pos = kNoPos; int fbi; Ray r; float tc = 0.0f;
        bool active = q < n;
        if (active && use_far) q = P.far_list[q];
        if (active && shading_point_repeats(P, depth, q)) {           // the parent cast this very ray: k_shade reads its verdict there
            n_shadow++; n_reused++;                                   // (every reflection path is a hit: 0 != 1e30f, raythread.cpp:227)
            active = false;
        }
        active = active && load_path<QUERY>(P, depth, q, slot, fbi, r, tc, pos) && pos != kNoPos;
        double r64[kRay64];
        TRay tr;
        uint32_t word = 0, bit = 0;
        if (active) {
            const DevShadowLight &L = P.slights[j];
            V3 position = vadd(r.o, vscale((double)tc, r.d));                                  // :360
            V3 lray = (L.type == CT_LIGHT_POINT) ? vsub(ld3(L.v), position) : ld3(L.v);        // :288 / :293
            Ray sr; sr.o = position; sr.d = lray; sr.t = kRayTInit;                            // :304 no offset, no t<=1 test
            tray_setup(tr, sr, P.bound, r64);
            n_shadow++;
            word = q * P.occ_words + (L.index >> 5); bit = L.index & 31u;
        }
        walk_or_park<kAnyHit, COUNT>(P, tr, r64, active, P.budget, ovf_idx, word, bit, n_parked, lc, sm,
                                     [&](int res, float, uint32_t) { if (res == kTravHit) atomicOr(&P.occ[word], 1u << bit); }, [](bool) {});
    }
    warp_add(&P.tot->rays_shadow, n_shadow);
    warp_add(&P.tot->rays_shadow_reused, n_reused);
    warp_add(&P.tot->rays_overflow, n_parked);
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// TraceRay's recursion step (raythread.cpp:369-373) for a path of `depth` whose hit record is final: does the path end here, or
// does it continue with the reflection ray {position, ReflectRay(-dir, normal), t = 0}?  Needs only the hit -- not the shadow
// verdicts -- so it runs in the hit kernel itself, in the warp that has just finished the walk (ray and hit are still in
// registers), and feeds k_bounce of the next depth.  WARP-LEVEL: every lane calls it, `active` = this lane holds such a path.
CT_DEV void emit_paths(const Params &P, int depth, bool active, uint32_t q, uint32_t slot, V3 o, V3 d, float tc, uint32_t pos, uint32_t &n_refl) {
    const int nxt = (depth & 1) ^ 1;
    bool emit = false;
    V3 position = {0, 0, 0}, rdir = {0, 0, 0};
    if (active) {
        float reflection = 0.0f;
        if (pos != kNoPos) reflection = P.materials[P.tris[pos].orig].reflection;
        const int remaining = P.max_depth - depth;                      // recursionDepth of this TraceRay call
        if (pos == kNoPos || remaining <= 0 || reflection <= 0.0f) {     // miss :385 / :369 (a NaN reflection recurses)
            P.term_level[slot] = (uint8_t)depth;
        } else {
            V3 p1, e1, e2;
            load_tri(P.tris, pos, p1, e1, e2);
            position = vadd(o, vscale((double)tc, d));                  // :360
            V3 nn = vcross(e1, e2);                                     // NormalOfSceneObject :337-339
            float dd = vdot(nn, d);
            V3 normal = (dd < 0.0f) ? nn : vneg(nn);                    // :341-345
            P.stack_refl[(size_t)depth * P.cap + slot] = reflection;
            rdir = reflect_ray(vneg(d), normal);                        // :372
            emit = true;
        }
    }
    // warp-aggregated append of the reflection rays to the next queue
    uint32_t mask = __ballot_sync(0xffffffffu, emit);
    if (mask) {
        uint32_t lane = threadIdx.x & 31u, leader = __ffs(mask) - 1, qbase = 0;
        if (lane == leader) qbase = atomicAdd(&P.sched->queue_count[depth + 1], (uint32_t)__popc(mask));
        qbase = __shfl_sync(0xffffffffu, qbase, leader);
        if (emit) {
            uint32_t nq = qbase + __popc(mask & ((1u << lane) - 1u));
            CT_CHECK(nq < P.cap && slot < P.cap);
            double2 *rb = reinterpret_cast<double2 *>(P.ray_buf[nxt] + 6ull * nq);
            rb[0] = make_double2(position.x, position.y);
            rb[1] = make_double2(position.z, rdir.x);
            rb[2] = make_double2(rdir.y, rdir.z);
            P.path_slot[nxt][nq] = slot;
            // would a hit with tclosest = 0 put the next shading point exactly here?  (not with a non-finite direction:
            // 0 * inf = NaN; and -0.0 + 0.0 = +0.0 changes a bit that a light at -0.0 could tell apart)
            const V3 again = vadd(position, vscale(0.0, rdir));
            const bool same = __double_as_longlong(again.x) == __double_as_longlong(position.x) &&
                              __double_as_longlong(again.y) == __double_as_longlong(position.y) &&
                              __double_as_longlong(again.z) == __double_as_longlong(position.z);
            P.parent_q[nxt][nq] = q | (same ? 0u : kNoReuse);
            n_refl++;
        }
    }
}

// The same step as a kernel of its own, for the paths whose hit record a hit kernel could not finish itself: the reflection
// paths k_bounce had parked (late_list; their hit came from k_overflow).  Depth >= 1 only, so its load_path needs no QUERY form.
__global__ void __launch_bounds__(kBlockThreads) k_emit(const __grid_constant__ Params P, int depth, int work_idx, const OvfRay *late_list, int ovf_bounce) {
    uint32_t n_refl = 0;
    const uint32_t n = min(P.sched->ovf_count[ovf_bounce], P.ovf_cap);
    while (true) {
        unsigned long long base = warp_fetch(&P.sched->work[work_idx]);
        if (base >= n) break;
        uint32_t q = (uint32_t)base + (threadIdx.x & 31u);
        bool active = q < n;
        if (active) q = late_list[q].target;
        uint32_t slot = q, pos = kNoPos; int fbi = 0;
        Ray r; float tc = 0.0f;
        r.o = {0, 0, 0}; r.d = {0, 0, 0};
        active = active && load_path(P, depth, q, slot, fbi, r, tc, pos);
        emit_paths(P, depth, active, q, slot, r.o, r.d, tc, pos, n_refl);
    }
    warp_add(&P.tot->rays_reflection, n_refl);
}

// TraceRay's local colour (raythread.cpp:359-366) for the paths alive at `depth`; the shadow verdicts were computed
// by k_shadow (+ k_overflow).
template <bool QUERY = false>
__global__ void __launch_bounds__(kBlockThreads) k_shade(const __grid_constant__ Params P, int depth, int work_idx) {
    const uint32_t n = depth == 0 ? depth0_count(P) : P.sched->queue_count[depth];
    while (true) {
        unsigned long long base = warp_fetch(&P.sched->work[work_idx]);
        if (base >= n) break;
        uint32_t q = (uint32_t)base + (threadIdx.x & 31u);
        uint32_t slot = q, pos = kNoPos; int fbi = 0;
        Ray r; float tc = 0.0f;
        if (!(q < n && load_path<QUERY>(P, depth, q, slot, fbi, r, tc, pos))) continue;
        uint32_t *sc = P.stack_color + (size_t)depth * P.cap + slot;
        if (pos == kNoPos) {                                           // miss (depth 0 only): raythread.cpp:385
            if (depth == 0) store_pixel(P, slot, fbi, P.background);
            *sc = P.background;
            continue;
        }
        V3 p1, e1, e2;
        load_tri(P.tris, pos, p1, e1, e2);
        const ct_material mat = P.materials[P.tris[pos].orig];
        V3 position = vadd(r.o, vscale((double)tc, r.d));              // :360
        V3 nn = vcross(e1, e2);                                         // NormalOfSceneObject :337-339
        float dd = vdot(nn, r.d);
        V3 normal = (dd < 0.0f) ? nn : vneg(nn);                        // :341-345
        V3 view = vneg(r.d);
        // ---- ComputeLighting :275-327, lights in file order, fp32 accumulator
        float intensity = 0.0f;
        const uint32_t *occ = occlusion_source(P, depth, q);
        uint32_t occ_word = 0;
        for (uint32_t i = 0; i < P.n_lights; i++) {
            const DevLight &L = P.lights[i];
            float li = L.intensity;
            if ((i & 31u) == 0) occ_word = occ[i >> 5];
            if (L.type == CT_LIGHT_AMBIENT) { intensity = __fadd_rn(intensity, li); continue; }
            if ((occ_word >> (i & 31u)) & 1u) continue;                  // :306 shadowed
            V3 lray = (L.type == CT_LIGHT_POINT) ? vsub(ld3(L.pos), position) : ld3(L.dir);
            float ndl = vdot(normal, lray);                              // :310
            if (ndl > 0.0f)
                intensity = __fadd_rn(intensity, __fdiv_rn(__fmul_rn(li, ndl), __fmul_rn(vmag(normal), vmag(lray))));
            if (mat.specular != -1) {                                    // :316
                V3 refl = reflect_ray(lray, normal);
                float rdv = vdot(refl, view);
                if (rdv > 0.0f) {                                        // :319-321 double pow, += rounds to float
                    float qv = __fdiv_rn(rdv, __fmul_rn(vmag(refl), vmag(view)));
                    intensity = specular_add(intensity, li, qv, mat.specular);
                }
            }
        }
        uint32_t local = shade_color(mat.color, intensity);
        *sc = local;
        // a depth-0 path that ends here (:369) is the pixel; longer chains are blended by k_resolve
        if (depth == 0 && (P.max_depth <= 0 || mat.reflection <= 0.0f)) store_pixel(P, slot, fbi, local);
    }
}

// Closest "hit" of the reflection rays {position, reflected, t = 0} (raythread.cpp:373).
template <bool COUNT>
__global__ void __launch_bounds__(kBlockThreads, kMinBlocks) k_bounce(const __grid_constant__ Params P, int depth, int work_idx, int ovf_idx) {
    LocalCount lc;
    uint32_t n_parked = 0, n_refl = 0;
    uint32_t *const sm = nullptr;                                     // (a first-line walk keeps its lists in local memory, traverse_wide)
    const uint32_t n = P.sched->queue_count[depth];
    const int cur = depth & 1;
    while (true) {
        unsigned long long base = warp_fetch(&P.sched->work[work_idx]);
        if (base >= n) break;
        uint32_t q = (uint32_t)base + (threadIdx.x & 31u);
        bool active = q < n;
        bool far = false;            // this path needs shadow rays of its own (its shading point is not, or may not be, its parent's)
        bool parked = false;
        double r64[kRay64];
        TRay r;
        if (active) {
            const double2 *rb = reinterpret_cast<const double2 *>(P.ray_buf[cur] + 6ull * q);
            double2 a = rb[0], b = rb[1], c = rb[2];
            Ray ray;
            ray.o = {a.x, a.y, b.x}; ray.d = {b.y, c.x, c.y}; ray.t = 0.0f;
            tray_setup(r, ray, P.bound, r64);
            clear_occ(P, q);
        }
        walk_or_park<kFirstLine, COUNT>(P, r, r64, active, P.budget, ovf_idx, q, 0u, n_parked, lc, sm,
            [&](int, float tc, uint32_t pos) {                          // found is always true: 0 != 1e30f (:227)
                P.hitb_t[q] = tc;
                P.hitb_pos[q] = (pos == kNoPos) ? P.pos_of_tri0 : pos;
                far = tc != 0.0f || (P.parent_q[cur][q] & kNoReuse);
            },
            [&](bool p) {
                far = true;                                             // k_overflow answers later: let k_shadow look at the path
                parked = p;
            });
        // the recursion step of the paths whose hit is final (parked ones: k_emit after k_overflow)
        const bool fin = q < n && !parked;
        uint32_t pslot = 0, ppos = kNoPos; float ptc = 0.0f;
        if (fin) { pslot = P.path_slot[cur][q]; ptc = P.hitb_t[q]; ppos = P.hitb_pos[q]; }
        emit_paths(P, depth, fin, q, pslot, {r64[0], r64[1], r64[2]}, {r64[3], r64[4], r64[5]}, ptc, ppos, n_refl);
        // warp-aggregated append to the depth's far list (see shading_point_repeats: the others repeat their parent's shading point)
        if (P.reuse_shadow) {
            const uint32_t mask = __ballot_sync(kFullMask, far);
            if (mask) {
                const uint32_t lane = threadIdx.x & 31u, leader = __ffs(mask) - 1;
                uint32_t fbase = 0;
                if (lane == leader) fbase = atomicAdd(&P.sched->far_count[depth], (uint32_t)__popc(mask));
                fbase = __shfl_sync(kFullMask, fbase, leader);
                if (far) P.far_list[fbase + __popc(mask & ((1u << lane) - 1u))] = q;
            }
        }
    }
    warp_add(&P.tot->rays_overflow, n_parked);
    warp_add(&P.tot->rays_reflection, n_refl);
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// Parked rays (see the file header).  Both early-exit modes have an answer that does not depend on the visit
// order, because ray.t never changes before the exit, so the set of boxes that pass is fixed:
//   kAnyHit     occluded  <=>  SOME triangle reachable through passing boxes has a bary pass with 1e-4 < t < 1e30;
//   kFirstLine  closestIndex = the bary-passing reachable triangle that the DFS meets first = the one with the
//               smallest leaf position where leaf positions increase along the DFS (BuildBVH hands the left child the
//               lower part of the parent's index range, bvh.cpp:70-97).  A caller's tree need not: upload checks it
//               (bvh_depth), and on a tree without it first-line rays are never parked (first_line_budget).
// Tests the triangles of an accepted leaf for a parked ray.  kAnyHit: 1 if one of them occludes, else 0;
// kFirstLine: the first (lowest) leaf position with a barycentric pass, else kNoPos.
template <TraverseMode MODE, bool COUNT>
CT_DEV uint32_t overflow_leaf(const Params &P, const TRay &r, uint32_t first, uint32_t cnt, LocalCount &lc) {
    for (uint32_t k = 0; k < cnt; k++) {
        uint32_t pos = first + k;
        if (COUNT) lc.tri++;
        const TriHit th = leaf_triangle<MODE == kAnyHit, COUNT>(P, r, pos, lc);
        if (!th.hit) continue;
        if (MODE == kAnyHit) { if (th.t > kEps && th.t < kRayTInit) return 1u; }
        else return pos;                                      // later positions of this leaf are larger
    }
    return MODE == kAnyHit ? 0u : kNoPos;
}

template <TraverseMode MODE>
CT_DEV uint32_t overflow_merge(uint32_t a, uint32_t b) { return MODE == kAnyHit ? (a | b) : min(a, b); }

template <TraverseMode MODE>
CT_DEV void overflow_store(const Params &P, const OvfRay &o, uint32_t res) {
    if (MODE == kAnyHit) {
        if (res) atomicOr(&P.occ[o.target], 1u << o.bit);
    } else {
        P.hitb_t[o.target] = (res == kNoPos) ? kFinf : 0.0f;          // raythread.cpp:204 / first line pass
        P.hitb_pos[o.target] = (res == kNoPos) ? P.pos_of_tri0 : res;
    }
}

constexpr int kWarpStack = 1024;         // pending interior nodes of one ray in the warp-cooperative pass
constexpr uint32_t kWarpBudget = 4096;       // default node visits before a ray is handed to the grid-wide pass

// Parked rays, pass 1: one WARP per ray -- the 32 lanes pop up to 32 pending interior nodes from a shared-memory
// stack, test their child pairs, test accepted leaves on the spot and push accepted interior children back.
// A ray whose stack outgrows kWarpStack, that needs more than P.warp_budget node visits or whose origin is so far
// outside the scene that every box passes (the rays described in the header: ~1M visits) goes to k_overflow_huge.
template <TraverseMode MODE, bool COUNT>
__global__ void __launch_bounds__(kOvfThreads) k_overflow(const __grid_constant__ Params P, int ovf_idx) {
    const uint32_t n = min(P.sched->ovf_count[ovf_idx], P.ovf_cap);
    if (n == 0) return;
    LocalCount lc;
    const uint32_t lane = threadIdx.x & 31u;
    __shared__ uint32_t wstack[kOvfThreads / 32][kWarpStack];
    uint32_t *stk = wstack[threadIdx.x >> 5];
    while (true) {
        uint32_t idx = 0;
        if (lane == 0) idx = atomicAdd(&P.sched->ovf_cursor[ovf_idx], 1u);
        idx = __shfl_sync(kFullMask, idx, 0);
        if (idx >= n) break;
        const OvfRay &o = P.ovf[idx];
        Ray ray; ray.o = ld3(o.o); ray.d = ld3(o.d); ray.t = (MODE == kAnyHit) ? kRayTInit : 0.0f;
        double r64[kRay64];
        TRay r;
        tray_setup(r, ray, P.bound, r64);             // every lane holds the same ray
        uint32_t res = MODE == kAnyHit ? 0u : kNoPos;
        // An origin this far outside the scene (a shading point 2^32 ray lengths away, SURVEY 0.4) makes all slab
        // quotients of an axis round to the same float: every box passes and no filter can help.
        bool too_big = !r.filt || (double)r.om > 0x1p20 * fmax(fmax(P.bound[0], P.bound[1]), P.bound[2]);
        if (COUNT && lane == 0 && !too_big) lc.box++;
        if (!too_big && exact_root(P, r64, r.t)) {
            if (P.root_cnt > 0) {
                if (lane == 0) res = overflow_leaf<MODE, COUNT>(P, r, P.root_ref, P.root_cnt, lc);
            } else {
                if (lane == 0) stk[0] = P.root_ref;
                __syncwarp();
                uint32_t sp = 1, visits = 0;
                while (sp > 0) {
                    const uint32_t take = min(sp, 32u);
                    sp -= take;
                    uint32_t n_out = 0, out_a = 0, out_b = 0;
                    if (lane < take) {
                        const uint32_t pid = stk[sp + lane];
                        DevPair32 pr;
                        load_pair32(P.pairs32, pid, pr);
                        if (COUNT) lc.box += 2;
                        bool hit_l, hit_r; float lo, hi;
                        pair_accept<COUNT>(P, r, pid, pr, hit_l, hit_r, lo, hi, lc);
                        if (hit_l) {
                            if (pr.l_cnt > 0) res = overflow_merge<MODE>(res, overflow_leaf<MODE, COUNT>(P, r, pr.l_ref, pr.l_cnt, lc));
                            else { out_a = pr.l_ref; n_out = 1; }
                        }
                        if (hit_r) {
                            if (pr.r_cnt > 0) res = overflow_merge<MODE>(res, overflow_leaf<MODE, COUNT>(P, r, pr.r_ref, pr.r_cnt, lc));
                            else { if (n_out) out_b = pr.r_ref; else out_a = pr.r_ref; n_out++; }
                        }
                    }
                    __syncwarp();                     // every lane has read its entry before the pushes below
                    if (MODE == kAnyHit && __any_sync(kFullMask, res != 0u)) break;
                    uint32_t incl = n_out;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { uint32_t v = __shfl_up_sync(kFullMask, incl, d); if ((int)lane >= d) incl += v; }
                    const uint32_t total = __shfl_sync(kFullMask, incl, 31);
                    visits += take;
                    if (sp + total > (uint32_t)kWarpStack || visits > P.warp_budget) { too_big = true; break; }
                    const uint32_t at = sp + incl - n_out;
                    if (n_out > 0) stk[at] = out_a;
                    if (n_out > 1) stk[at + 1u] = out_b;
                    sp += total;
                    __syncwarp();
                }
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) res = overflow_merge<MODE>(res, __shfl_xor_sync(kFullMask, res, d));
        if (lane == 0) {
            if (too_big) {
                P.ovf_huge[atomicAdd(&P.sched->huge_count[ovf_idx], 1u)] = idx;
                if (MODE == kFirstLine) { P.hitb_t[o.target] = kFinf; P.hitb_pos[o.target] = kNoPos; }   // until k_overflow_huge finds a pass
            } else {
                overflow_store<MODE>(P, o, res);
            }
        }
    }
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// Is the leaf that holds a triangle REACHED by the reference's walk?  Every box on the way down must accept the ray:
// the leaf's own box, its ancestors' boxes, the root's.  `code` = 2 * pair + side of the leaf's box.
CT_DEV bool chain_accepts(const Params &P, double *r64, float ray_t, uint32_t code) {
    while (code != kNoPos) {
        const uint32_t pid = code >> 1;
        if (!box_accept(exact_child(P.pairs64, pid, code & 1u, r64), ray_t)) return false;
        code = P.pair_parent[pid];
    }
    return exact_root(P, r64, ray_t);
}

// Parked rays, pass 2 (what pass 1 gave up on).  Walking a tree in which every box passes level by level costs a
// grid-wide barrier per level; instead the whole grid tests ALL triangles against the ray at once and, for the few
// that pass, checks whether the reference's walk would have reached them at all (chain_accepts).  No barrier, and
// the answers are merged with idempotent atomics (OR into the occlusion mask / MIN of the leaf position).
template <TraverseMode MODE, bool COUNT>
__global__ void __launch_bounds__(256) k_overflow_huge(const __grid_constant__ Params P, int ovf_idx) {
    const uint32_t nh = P.sched->huge_count[ovf_idx];
    if (nh == 0) return;
    LocalCount lc;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, n_threads = gridDim.x * blockDim.x;
    for (uint32_t h = 0; h < nh; h++) {
        const OvfRay &o = P.ovf[P.ovf_huge[h]];
        Ray ray; ray.o = ld3(o.o); ray.d = ld3(o.d); ray.t = (MODE == kAnyHit) ? kRayTInit : 0.0f;
        double r64[kRay64];
        TRay r;
        tray_setup(r, ray, P.bound, r64);
        for (uint32_t pos = tid; pos < P.n_tri; pos += n_threads) {
            if (MODE == kAnyHit && (*(volatile uint32_t *)&P.occ[o.target] >> o.bit) & 1u) break;      // already occluded
            if (MODE == kFirstLine && *(volatile uint32_t *)&P.hitb_pos[o.target] < pos) break;        // a lower position already passed
            if (COUNT) lc.tri++;
            const TriHit th = leaf_triangle<MODE == kAnyHit, COUNT>(P, r, pos, lc);
            if (!th.hit) continue;
            if (MODE == kAnyHit && !(th.t > kEps && th.t < kRayTInit)) continue;
            if (!chain_accepts(P, r64, r.t, P.tri_parent[pos])) continue;
            if (MODE == kAnyHit) atomicOr(&P.occ[o.target], 1u << o.bit);
            else { atomicMin(&P.hitb_pos[o.target], pos); P.hitb_t[o.target] = 0.0f; }
        }
    }
    if (COUNT) { warp_add(&P.tot->box_tests, lc.box); warp_add(&P.tot->tri_tests, lc.tri); warp_add(&P.tot->box_exact, lc.box_exact); warp_add(&P.tot->tri_exact, lc.tri_exact); }
}

// Unwind TraceRay's recursion (raythread.cpp:375-379) for pixels whose chain went past depth 0.
template <bool QUERY = false>
__global__ void __launch_bounds__(256) k_resolve(const __grid_constant__ Params P) {
    const uint32_t n = depth0_count(P);
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const uint32_t slot = own_slot(P, q);
        int x, y, fbi;
        if (!slot_pixel<QUERY>(P, slot, x, y, fbi)) continue;
        int lvl = P.term_level[slot];
        if (lvl == 0) continue;                              // already stored by k_shade
        uint32_t color = P.stack_color[(size_t)lvl * P.cap + slot];
        for (int d = lvl - 1; d >= 0; d--)
            color = blend_color(P.stack_color[(size_t)d * P.cap + slot], color, P.stack_refl[(size_t)d * P.cap + slot]);
        store_pixel(P, slot, fbi, color);
    }
}

// settings.subsampling (raythread.cpp:512-531): after a traced pixel (x, y) the reference stores the average of its
// colour and the previously traced colour of the column (its own for the first row of the partition) one row
// below, at (x, y - 1).  Runs after every traced pixel of the tile has its final colour; a later store wins where
// the reference's sequential loop would overwrite (the always-traced last row of an even partition).
__global__ void __launch_bounds__(256) k_subsample(const __grid_constant__ Params P) {
    const uint32_t ss = P.supersample ? 4u : 0u;              // with supersampling a pixel owns 16 slots; its blended colour sits in the first
    const uint32_t n = depth0_count(P) >> ss;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t slot = own_slot(P, i << ss);
        int x, y, fbi;
        if (!slot_pixel(P, slot, x, y, fbi)) continue;
        const uint32_t pix = slot >> ss, blk = pix >> 5, lane = pix & 31u;
        const uint32_t iy = (blk / (uint32_t)P.blocks_x) * 4u + (lane >> 3);
        const uint32_t color = P.final_color[slot];
        uint32_t last = color;                                                 // :513-514
        if (iy > 0) {
            const uint32_t py = iy - 1u, ix = (blk % (uint32_t)P.blocks_x) * 8u + (lane & 7u);
            last = P.final_color[((((py >> 2) * (uint32_t)P.blocks_x + (ix >> 3)) << 5) + ((py & 3u) << 3) + (ix & 7u)) << ss];
        }
        uint32_t avg = 0;                                                      // :517-523: float (a + b) / 2, min 0xff, truncated
        for (int sh = 0; sh <= 16; sh += 8) avg |= ((((last >> sh) & 0xffu) + ((color >> sh) & 0xffu)) >> 1) << sh;
        const int col = x + P.W / 2, row = P.H / 2 - (y - 1);                  // CanvasPutPixel(bitmap, {x, y-1}, avgColor) :524
        if (row >= 0 && row < P.H && col >= 0 && col < P.W) P.fb_out[row * P.W + col] = avg;
    }
}

// settings.supersampling (raythread.cpp:460-505): the 16 samples of a pixel are folded into its colour one after the
// other -- colour -= colour/8; colour += sample/8 per channel in float, truncated to uint8 after every sample (:486-497).
__global__ void __launch_bounds__(256) k_supersample(const __grid_constant__ Params P) {
    const uint32_t n = depth0_count(P) >> 4;                                  // chunks hold whole pixels (32 or 64 slots)
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t slot = own_slot(P, i << 4);
        int x, y, fbi;
        if (!slot_pixel(P, slot, x, y, fbi)) continue;
        uint32_t color = P.final_color[slot];
        for (uint32_t k = 1; k < 16u; k++) {
            const uint32_t temp = P.final_color[slot + k];
            uint32_t out = 0;
            for (int sh = 0; sh <= 16; sh += 8) {
                float c = (float)((color >> sh) & 0xffu), t = (float)((temp >> sh) & 0xffu);
                c = __fsub_rn(c, __fdiv_rn(c, 8.0f));
                c = __fadd_rn(c, __fdiv_rn(t, 8.0f));
                out |= to_u8(c) << sh;
            }
            color = out;
        }
        const int col = x + P.W / 2, row = P.H / 2 - y;
        if (row >= 0 && row < P.H) P.fb_out[row * P.W + col] = color;          // with subsampling a row PutPixel drops is still traced
        if (P.subsample) P.final_color[slot] = color;                          // the pixel's colour, for k_subsample (runs after this kernel)
    }
}

// ---- KAT kernels -----------------------------------------------------------------------------------------
__global__ void k_debug_closest(const __grid_constant__ Params P, uint32_t n, const double *org, const double *dir,
                                const float *t0, uint32_t *found, uint32_t *index, float *tclosest) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;                           // the traversals are warp-synchronous: every lane calls both
    Ray r;
    r.t = 1.0f;
    double r64[kRay64];
    TRay tr;
    if (active) {
        r.o = ld3(org + 3ull * i); r.d = ld3(dir + 3ull * i); r.t = t0[i];
        tray_setup(tr, r, P.bound, r64);
    }
    LocalCount lc; float tc, tc2; uint32_t pos, pos2;
    const bool first_line = r.t == 0.0f;
    bool f = traverse_early_any<kFirstLine, false>(P, tr, active && first_line, 0xffffffffu, tc, pos, lc, nullptr) == kTravHit;
    bool f2 = traverse_closest<false>(P, tr, active && !first_line, tc2, pos2, lc) == kTravHit;
    if (!active) return;
    if (!first_line) { f = f2; tc = tc2; pos = pos2; }
    if (found) found[i] = f ? 1u : 0u;
    if (index) index[i] = (pos == kNoPos) ? 0u : P.tris[pos].orig;
    if (tclosest) tclosest[i] = tc;
}

// ---- ray queries (ct_gpu_trace_rays; ct_gpu_debug_early / ct_gpu_debug_primary are host-memory wrappers of the same path) ----
// Thread t walks ray t, in the caller's order.  Every answer -- the walk's own, and those of the parked rays that the real
// k_overflow / k_overflow_huge, k_primary_long / k_primary_split deliver -- goes to the ray's hit record or occlusion word at the
// CALLER's index i (the parking target), and k_ray_results turns these into the outputs at index i.

// Shadow rays (kAnyHit, ray.t = 1e30f: P.occ[i] = occluded) and reflection rays (kFirstLine, ray.t = 0: the hit record
// P.hitb_t[i] / P.hitb_pos[i] as k_bounce writes it) through walk_or_park as k_shadow / k_bounce run theirs; the parked ones are
// answered into the same words by k_overflow / k_overflow_huge.  path[i] (may be NULL): 0 own walk, 1 parked, 3 finished in place.
// (__maxnreg__: left to itself ptxas gives the first-line walk 80 registers and spills; with up to 96 neither walk spills)
template <TraverseMode MODE>
__global__ void __maxnreg__(96) k_debug_early(const __grid_constant__ Params P, uint32_t n, const double *org, const double *dir,
                                              uint32_t *path) {
    __shared__ uint32_t walk_sm[kWalkWords * kBlockThreads];          // launched with kBlockThreads threads per block, like k_shadow
    uint32_t *const sm = MODE == kAnyHit ? walk_sm + threadIdx.x : nullptr;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;                                         // walk_or_park is warp-level: every lane calls it
    LocalCount lc;
    double r64[kRay64];
    TRay tr;
    if (active) {
        Ray r;
        r.o = ld3(org + 3ull * i); r.d = ld3(dir + 3ull * i); r.t = MODE == kAnyHit ? kRayTInit : 0.0f;
        tray_setup(tr, r, P.bound, r64);
    }
    uint32_t n_parked = 0;
    const int how = walk_or_park<MODE, false>(P, tr, r64, active, P.budget, 0, i, 0u, n_parked, lc, sm,
        [&](int res, float tc, uint32_t pos) {
            if (MODE == kAnyHit) P.occ[i] = res == kTravHit ? 1u : 0u;
            else { P.hitb_t[i] = tc; P.hitb_pos[i] = (pos == kNoPos) ? P.pos_of_tri0 : pos; }     // found is always true (:227)
        }, [&](bool parked) { if (MODE == kAnyHit && parked) P.occ[i] = 0u; });      // k_overflow ORs the verdict in
    if (active && path) path[i] = (uint32_t)how;
}

// Primary rays (ray.t = 1e30f) through primary_walk_or_park as k_primary runs its rays, path q = slot = i: the hit record goes to
// P.hit0_t[i] / P.hit0_pos[i], that of a parked ray from the real k_primary_long / k_primary_split.  path[i] (may be NULL): 0 own
// walk, 1 parked, 3 finished in place (k_primary_split rewrites its rays' codes through P.split_path).
template <bool PARK>
__global__ void __launch_bounds__(kBlockThreads, kMinBlocks) k_debug_primary(const __grid_constant__ Params P, uint32_t n, const double *org,
                                                                             const double *dir, uint32_t *path) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;                                         // primary_walk_or_park is warp-level: every lane calls it
    LocalCount lc;
    double r64[kRay64];
    TRay r;
    if (active) {
        Ray ray;
        ray.o = ld3(org + 3ull * i); ray.d = ld3(dir + 3ull * i); ray.t = kRayTInit;
        tray_setup(r, ray, P.bound, r64);
    }
    uint32_t n_parked = 0;
    int res; float tc; uint32_t pos;
    const int how = primary_walk_or_park<false, PARK>(P, r, r64, active, i, i, n_parked, lc, res, tc, pos);
    if (!active) return;
    if (path) path[i] = (uint32_t)how;
    if (how != kParked) store_primary_hit(P, i, i, -1, res == kTravHit, tc, pos);
}

// Every ray's outputs from its hit record / occlusion word, after the parked rays' kernels (any output may be NULL):
//   kClosest    found, ClosestIntersection's closestIndex and tclosest (P.hit0_*: pos_of_tri0 for a hit without a closestIndex);
//   kFirstLine  found = 1 (0 != 1e30f, raythread.cpp:227), the first pass's index, tclosest 0 or FINF (P.hitb_*);
//   kAnyHit     found = occluded, index 0 (P.occ bit 0).
// path: 2 for the rays k_overflow handed to k_overflow_huge.
__global__ void k_ray_results(const __grid_constant__ Params P, int mode, uint32_t n, uint32_t *found, uint32_t *index, float *tclosest,
                              uint32_t *path) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (path && i < P.sched->huge_count[0]) path[P.ovf[P.ovf_huge[i]].target] = 2u;
    if (i >= n) return;
    if (mode == kAnyHit) {
        if (found) found[i] = P.occ[i] & 1u;
        if (index) index[i] = 0u;
        return;
    }
    const uint32_t pos = mode == kClosest ? P.hit0_pos[i] : P.hitb_pos[i];
    if (found) found[i] = (mode == kFirstLine || pos != kNoPos) ? 1u : 0u;
    if (index) index[i] = pos == kNoPos ? 0u : P.tris[pos].orig;
    if (tclosest) tclosest[i] = mode == kClosest ? P.hit0_t[i] : P.hitb_t[i];
}

__global__ void k_debug_primitives(uint32_t n,const double *org, const double *dir, float *ray_t, const double *tri,
                                   const double *bmin, const double *bmax, uint32_t *tri_hit, uint32_t *box_hit,
                                   uint32_t *filter_out, double bound_scale, bool tri_filter) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Ray r;
    r.o = ld3(org + 3ull * i); r.d = ld3(dir + 3ull * i); r.t = ray_t[i];
    double mn[3] = {bmin[3ull * i], bmin[3ull * i + 1], bmin[3ull * i + 2]};
    double mx[3] = {bmax[3ull * i], bmax[3ull * i + 1], bmax[3ull * i + 2]};
    const bool exact = intersect_aabb(r, mn, mx);
    box_hit[i] = exact ? 1u : 0u;
    if (filter_out) {
        // the certified filter on the same box: bit 0 exact verdict, bits 1-2 filter (0 undecided, 1 accept, 2 reject),
        // bit 3 = the filter was usable for this ray.  A certain verdict that contradicts bit 0 is a soundness bug.
        double bnd[3];
        bool ordered = true;
        for (int k = 0; k < 3; k++) {
            bnd[k] = fmax(fabs(mn[k]), fabs(mx[k])) * bound_scale;
            ordered = ordered && (mn[k] <= mx[k]) && isfinite(mn[k]) && isfinite(mx[k]);
        }
        if (!ordered) bnd[0] = bnd[1] = bnd[2] = INFINITY;
        double r64[kRay64];
        TRay tr;
        tray_setup(tr, r, bnd, r64);
        uint32_t f = 0;
        if (tr.filt) {
            const float fmn[3] = {(float)mn[0], (float)mn[1], (float)mn[2]}, fmx[3] = {(float)mx[0], (float)mx[1], (float)mx[2]};
            BoxBracket b = box_filter(tr, fmn, fmx);
            if (bracket_geom_no(b) || bracket_t_no(b, r.t)) f = 2;
            else if (bracket_geom_yes(b) && bracket_t_yes(b, r.t)) f = 1;
            BoxTimes e = box_times(r, mn, mx);
            bool inside = b.near_lo <= e.tmin && e.tmin <= b.near_hi && b.far_lo <= e.tmax && e.tmax <= b.far_hi;
            if (!inside) f |= 8u;                                  // bracket does not contain the reference's floats: bug
        }
        // the division-free evaluation used for undecided tests must give the literal arithmetic's verdict and floats
        {
            const BoxTimes lit = box_times(r, mn, mx), rec = box_times(r64, mn, mx);
            const bool same = (lit.tmin == rec.tmin || (lit.tmin != lit.tmin && rec.tmin != rec.tmin)) &&
                              (lit.tmax == rec.tmax || (lit.tmax != lit.tmax && rec.tmax != rec.tmax));
            if (!same || box_accept(rec, r.t) != exact) f |= 16u;
        }
        uint32_t out = (exact ? 1u : 0u) | ((f & 3u) << 1) | (tr.filt ? 8u : 0u) | ((f & 8u) ? 16u : 0u) | ((f & 16u) ? 32u : 0u);
        if (tri_filter) {
            // the certified triangle filter on the same (ray, triangle), with the magnitudes the upload would store:
            // bit 8 = reference returns true, bit 9 = ... and the hit would occlude a shadow ray (1e-4 < t < 1e30),
            // bit 10 / 11 = tri_filter_miss<false> / <true> say "certainly no effect", bit 12 = filter usable
            const V3 q1 = ld3(tri + 9ull * i), q2 = ld3(tri + 9ull * i + 3), q3 = ld3(tri + 9ull * i + 6);
            const V3 e1 = vsub(q2, q1), e2 = vsub(q3, q1);
            float tt = 0.0f;
            const bool th = intersect_triangle(r, q1, e1, e2, &tt);
            const double k1 = fmax(fmax(fabs(e1.x), fabs(e1.y)), fabs(e1.z)), k2 = fmax(fmax(fabs(e2.x), fabs(e2.y)), fabs(e2.z));
            const double k3 = fmax(fmax(fabs(q1.x), fabs(q1.y)), fabs(q1.z));
            const bool in_range = k1 >= 0x1p-30 && k1 <= 0x1p30 && k2 >= 0x1p-30 && k2 <= 0x1p30 && k3 <= 0x1p40;
            const float4 t0 = make_float4((float)q1.x, (float)q1.y, (float)q1.z, __double2float_ru(k3));
            const float4 t1 = make_float4((float)e1.x, (float)e1.y, (float)e1.z, in_range ? __double2float_ru(k1) : NAN);
            const float4 t2 = make_float4((float)e2.x, (float)e2.y, (float)e2.z, __double2float_ru(k2));
            const bool m0 = tr.tfilt && tri_filter_miss<false>(tr, t0, t1, t2), m1 = tr.tfilt && tri_filter_miss<true>(tr, t0, t1, t2);
            out |= (th ? 1u << 8 : 0u) | ((th && tt > kEps && tt < kRayTInit) ? 1u << 9 : 0u) | (m0 ? 1u << 10 : 0u) | (m1 ? 1u << 11 : 0u) | (tr.tfilt ? 1u << 12 : 0u);
        }
        filter_out[i] = out;
    }
    V3 p1 = ld3(tri + 9ull * i), p2 = ld3(tri + 9ull * i + 3), p3 = ld3(tri + 9ull * i + 6);
    float t;
    bool hit = intersect_triangle(r, p1, vsub(p2, p1), vsub(p3, p1), &t);
    if (hit && t > kEps) r.t = macro_min(r.t, t);
    tri_hit[i] = hit ? 1u : 0u;
    ray_t[i] = r.t;
}

// The shading arithmetic of k_shade / k_resolve on n independent cases (ct_gpu_debug_shading); a NULL output skips its family.
__global__ void k_debug_shading(uint32_t n, const uint32_t *color, const float *intensity, uint32_t *shaded,
                                const uint32_t *lc, const uint32_t *rc, const float *reflection, uint32_t *blended,
                                const float *x, const int32_t *e, double *pw, const float *acc, const float *li, float *acc_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (shaded) shaded[i] = shade_color(color[i], intensity[i]);
    if (blended) blended[i] = blend_color(lc[i], rc[i], reflection[i]);
    if (pw) pw[i] = pow_int((double)x[i], e[i]);
    if (acc_out) acc_out[i] = specular_add(acc[i], li[i], x[i], e[i]);
}

}  // namespace
