// ct_bvh_build.cuh -- the reference's BuildBVH (bvh.cpp:16-120) on the device: ct_gpu_build_bvh.
// Part of the single translation unit ct_gpu.cu (everything lives in its anonymous namespace).
//
// Output is node for node and index for index the reference's tree (ct_bvh.cpp explains why that matters).  The build is
// level-synchronous: every level of the tree is one pass of a handful of kernels over all n positions of the index array,
// and the host loops until a level makes no split (no depth bound is assumed).  Per level:
//   k_bb_pred      the partition predicate float(centroid[axis]) < split of every position inside a node that is split;
//   scan           one exclusive prefix sum over all n positions: smalls before position p inside its node = S[p] - S[first];
//   k_bb_nodes     k (smalls) per node, the split decision, and one flag per split for the children's numbering;
//   scan           over the level's nodes: children of the m-th split are level_end + 2 m, + 1 (temporary ids, level order);
//   k_bb_children  the children's ranges;
//   k_bb_pair      who pairs with whom in the in-place partition (bvh.cpp:70-81);
//   k_bb_scatter   every entry to the place the closed form of that partition gives it (split_node_parallel in
//                  ct_bvh.cpp, tools/partition_closed_form.py), including the permutation of a node that then declines
//                  to split;
//   k_bb_bounds / k_bb_finish   the children's bounds (UpdateNodeBounds, bvh.cpp:30-49) by ordered reductions, and their
//                  axis and split plane.
// Then the reference's numbering comes from the shape alone (tools/bvh_numbering_check.py): interior counts bottom-up,
// pre-order ranks top-down, left(X) = 1 + 2 * rank(X), and one scatter to the final indices.
//
// There is no small-node cut-off and no compaction: every level is processed by the same kernels over all n positions, finished
// ones included (k_bb_scatter copies their 64-byte records again), so the build moves O(n * depth) bytes -- about 110 MB per
// level for 868k triangles, 29 levels for the dragon-class scene.  A deep comb inside a large scene pays that once per level.
//
// Rounding points (all reproduced; -fmad=false and explicit _rn intrinsics keep them):
//   centroid = (double)0.3333f * ((p1 + p2) + p3) in fp64; the partition reads float(centroid[axis])       bvh.cpp:112
//   bounds start at (double)1e30f / (double)-1e30f and fold with a < b ? a : b (ties: the later operand)   bvh.cpp:30-49
//   axis 1 if ext[1] > ext[0]; axis 2 if ext[2] > (double)(float)ext[axis]                                 bvh.cpp:61-65
//   split = (float)min[axis] + (float)ext[axis] * 0.5f in fp32; predicate strict <                        bvh.cpp:67,73
#pragma once

#include "ct_layout.cuh"

namespace {

constexpr uint32_t kBbThreads = 256;          // threads per CTA of every build kernel
constexpr uint32_t kBbScanTile = 1024;        // entries per CTA of the prefix sum (4 per thread)
constexpr uint32_t kBbChunk = 256;            // positions per warp in k_bb_bounds (8 rounds of 32)
constexpr uint32_t kBbNone = 0xffffffffu;     // owner of a position whose node is final

// one triangle, moved with the permutation: its per-axis vertex min / max (the fold of its three vertices), float(centroid)
// and its index
struct __align__(16) BbRec { double mn[3], mx[3]; float c[3]; uint32_t idx; };
static_assert(sizeof(BbRec) == 64, "BbRec is one 64-byte record");

// a node under construction (temporary id = level order)
struct BbNode {
    double mn[3], mx[3];
    uint32_t first, count;
    uint32_t left;            // temporary id of the left child; 0 = leaf (the root is never a child)
    uint32_t k;               // smalls of the partition
    uint32_t n_pairs;         // larges in [0, k) = smalls in [k, count): the swaps of the partition
    uint32_t hi;              // last entry of the untouched middle (local)
    uint32_t axis;
    float split;
};

// mymath.h:11,15 macro semantics: on ties the later operand wins (it matters for +0.0 / -0.0)
__device__ __forceinline__ double bb_lo(double a, double b) { return (a < b) ? a : b; }
__device__ __forceinline__ double bb_hi(double a, double b) { return (a > b) ? a : b; }

__device__ __forceinline__ uint32_t bb_tid() { return blockIdx.x * blockDim.x + threadIdx.x; }
__device__ __forceinline__ uint32_t bb_stride() { return gridDim.x * blockDim.x; }

// ---- exclusive prefix sum in place over a[0 .. m] (a[m] is an input of 0 and becomes the total) ------------------------
__global__ void __launch_bounds__(kBbThreads) k_bb_scan_reduce(const uint32_t *__restrict__ a, uint32_t m1, uint32_t *__restrict__ tile_sum) {
    __shared__ uint32_t red[kBbThreads / 32];
    const uint32_t base = blockIdx.x * kBbScanTile + threadIdx.x * 4u;
    uint32_t s = 0;
    for (uint32_t i = 0; i < 4u; i++) if (base + i < m1) s += a[base + i];
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31u) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (uint32_t w = 0; w < kBbThreads / 32; w++) t += red[w];
        tile_sum[blockIdx.x] = t;
    }
}

// block-wide exclusive scan of one value per thread; returns the exclusive prefix and sets *total
__device__ uint32_t bb_block_scan(uint32_t v, uint32_t *total) {
    __shared__ uint32_t warp_sum[kBbThreads / 32];
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    uint32_t x = v;
    for (int off = 1; off < 32; off <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, off); if (lane >= (uint32_t)off) x += y; }
    if (lane == 31u) warp_sum[w] = x;
    __syncthreads();
    uint32_t before = 0, all = 0;
    for (uint32_t i = 0; i < kBbThreads / 32; i++) { if (i < w) before += warp_sum[i]; all += warp_sum[i]; }
    __syncthreads();
    *total = all;
    return before + x - v;
}

// one CTA: exclusive scan of the tile sums, in place
__global__ void __launch_bounds__(kBbThreads) k_bb_scan_tiles(uint32_t *__restrict__ tile_sum, uint32_t n_tiles) {
    uint32_t carry = 0;
    for (uint32_t b = 0; b < n_tiles; b += kBbThreads * 4u) {
        uint32_t v[4], s = 0;
        for (uint32_t i = 0; i < 4u; i++) { const uint32_t j = b + threadIdx.x * 4u + i; v[i] = j < n_tiles ? tile_sum[j] : 0u; s += v[i]; }
        uint32_t total;
        uint32_t run = carry + bb_block_scan(s, &total);
        for (uint32_t i = 0; i < 4u; i++) { const uint32_t j = b + threadIdx.x * 4u + i; if (j < n_tiles) tile_sum[j] = run; run += v[i]; }
        carry += total;
    }
}

__global__ void __launch_bounds__(kBbThreads) k_bb_scan_down(uint32_t *__restrict__ a, uint32_t m1, const uint32_t *__restrict__ tile_sum) {
    const uint32_t base = blockIdx.x * kBbScanTile + threadIdx.x * 4u;
    uint32_t v[4], s = 0;
    for (uint32_t i = 0; i < 4u; i++) { v[i] = base + i < m1 ? a[base + i] : 0u; s += v[i]; }
    uint32_t total;
    uint32_t run = tile_sum[blockIdx.x] + bb_block_scan(s, &total);
    for (uint32_t i = 0; i < 4u; i++) if (base + i < m1) { a[base + i] = run; run += v[i]; }
}

// a[0 .. m) -> exclusive prefix sums, a[m] = total (a holds m + 1 entries, a[m] == 0 on entry)
cudaError_t bb_scan(uint32_t *a, uint32_t m, uint32_t *tile_sum, cudaStream_t st) {
    const uint32_t m1 = m + 1u, tiles = (m1 + kBbScanTile - 1u) / kBbScanTile;
    k_bb_scan_reduce<<<tiles, kBbThreads, 0, st>>>(a, m1, tile_sum);
    k_bb_scan_tiles<<<1, kBbThreads, 0, st>>>(tile_sum, tiles);
    k_bb_scan_down<<<tiles, kBbThreads, 0, st>>>(a, m1, tile_sum);
    return cudaGetLastError();
}

// ---- records, level 0 ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBbThreads) k_bb_init(const unsigned char *__restrict__ raw, uint32_t stride, uint32_t n,
                                                        BbRec *__restrict__ rec, uint32_t *__restrict__ own, BbNode *__restrict__ nodes) {
    const double third = (double)0.3333f;
    for (uint32_t k = bb_tid(); k < n; k += bb_stride()) {
        const double *v = reinterpret_cast<const double *>(raw + (size_t)k * stride);
        BbRec r;
        for (int a = 0; a < 3; a++) {
            r.mn[a] = bb_lo(bb_lo(v[a], v[3 + a]), v[6 + a]);     // the fold of the three vertices: its last minimum / maximum
            r.mx[a] = bb_hi(bb_hi(v[a], v[3 + a]), v[6 + a]);
            r.c[a] = __double2float_rn(__dmul_rn(third, __dadd_rn(__dadd_rn(v[a], v[3 + a]), v[6 + a])));
        }
        r.idx = k;
        rec[k] = r;
        own[k] = 0u;
    }
    if (bb_tid() == 0) {
        BbNode root{};
        root.first = 0; root.count = n;
        nodes[0] = root;
    }
}

// ---- one level ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool bb_splits(const BbNode &nd) { return nd.count > 2u; }      // bvh.cpp:54: a node of <= 2 is a leaf, unpermuted

__global__ void __launch_bounds__(kBbThreads) k_bb_pred(const BbRec *__restrict__ rec, const uint32_t *__restrict__ own,
                                                        const BbNode *__restrict__ nodes, uint32_t n, uint32_t *__restrict__ S) {
    for (uint32_t p = bb_tid(); p <= n; p += bb_stride()) {
        uint32_t small = 0;
        if (p < n && own[p] != kBbNone) {
            const BbNode &nd = nodes[own[p]];
            if (bb_splits(nd)) small = rec[p].c[nd.axis] < nd.split ? 1u : 0u;
        }
        S[p] = small;
    }
}

__global__ void __launch_bounds__(kBbThreads) k_bb_nodes(BbNode *__restrict__ nodes, uint32_t b, uint32_t e, const uint32_t *__restrict__ S,
                                                         uint32_t *__restrict__ before, uint32_t *__restrict__ NS) {
    for (uint32_t i = b + bb_tid(); i < e; i += bb_stride()) {
        BbNode &nd = nodes[i];
        uint32_t split = 0;
        if (bb_splits(nd)) {
            const uint32_t s0 = S[nd.first];
            nd.k = S[nd.first + nd.count] - s0;
            nd.n_pairs = nd.k - (S[nd.first + nd.k] - s0);
            nd.hi = nd.count - 1u;                                  // no pairs: the middle is all of [k, count)
            before[nd.first] = 0u;
            split = (nd.k != 0u && nd.k != nd.count) ? 1u : 0u;     // bvh.cpp:84-86
        }
        NS[i - b] = split;
    }
    if (bb_tid() == 0) NS[e - b] = 0u;
}

__global__ void __launch_bounds__(kBbThreads) k_bb_children(BbNode *__restrict__ nodes, uint32_t b, uint32_t e, const uint32_t *__restrict__ NS) {
    for (uint32_t i = b + bb_tid(); i < e; i += bb_stride()) {
        if (NS[i - b + 1] == NS[i - b]) continue;
        BbNode &nd = nodes[i];
        const uint32_t l = e + 2u * NS[i - b];
        nd.left = l;
        BbNode c{};
        c.first = nd.first; c.count = nd.k;
        nodes[l] = c;
        c.first = nd.first + nd.k; c.count = nd.count - nd.k;
        nodes[l + 1u] = c;
    }
}

__global__ void __launch_bounds__(kBbThreads) k_bb_pair(const uint32_t *__restrict__ own, BbNode *__restrict__ nodes, uint32_t n,
                                                        const uint32_t *__restrict__ S, uint32_t *__restrict__ ll_pos, uint32_t *__restrict__ before) {
    for (uint32_t p = bb_tid(); p < n; p += bb_stride()) {
        if (own[p] == kBbNone) continue;
        BbNode &nd = nodes[own[p]];
        if (!bb_splits(nd)) continue;
        const uint32_t q = p - nd.first, sm = S[p] - S[nd.first], k = nd.k;
        if (S[p + 1] != S[p]) {                                     // a small
            if (q >= k) {
                const uint32_t r = k - (sm + 1u);                   // smalls above q: its rank from the end
                if (r + 1u < nd.n_pairs) before[nd.first + r + 1u] = (r + 1u) + ((nd.count - k) - (q + 1u - (sm + 1u)));
                if (r + 1u == nd.n_pairs) nd.hi = q - 1u;
            }
        } else if (q < k) {
            ll_pos[nd.first + (q - sm)] = q;                        // larges before q: its rank among the left larges
        }
    }
}

__global__ void __launch_bounds__(kBbThreads) k_bb_scatter(const BbRec *__restrict__ rec, const uint32_t *__restrict__ own, const BbNode *__restrict__ nodes,
                                                           uint32_t n, const uint32_t *__restrict__ S, const uint32_t *__restrict__ ll_pos,
                                                           const uint32_t *__restrict__ before, BbRec *__restrict__ rec_out, uint32_t *__restrict__ own_out) {
    for (uint32_t p = bb_tid(); p < n; p += bb_stride()) {
        const uint32_t o = own[p];
        if (o == kBbNone || !bb_splits(nodes[o])) { rec_out[p] = rec[p]; own_out[p] = kBbNone; continue; }
        const BbNode nd = nodes[o];
        const uint32_t q = p - nd.first, sm = S[p] - S[nd.first], k = nd.k, cnt = nd.count;
        uint32_t dest;
        if (S[p + 1] != S[p]) {
            dest = q < k ? q : ll_pos[nd.first + k - (sm + 1u)];
        } else if (q < k) {
            dest = cnt - 1u - before[nd.first + (q - sm)];
        } else {
            const uint32_t above = k - sm;                          // smalls above q
            if (above < nd.n_pairs) dest = cnt - 1u - (above + 1u) - ((cnt - k) - (q + 1u - sm));
            else dest = q > k ? q - 1u : nd.hi;                     // the untouched middle, rotated left by one
        }
        rec_out[nd.first + dest] = rec[p];
        own_out[nd.first + dest] = nd.left ? nd.left + (dest < k ? 0u : 1u) : kBbNone;
    }
}

// Bounds of the nodes of a new level: warp w folds positions [w C, (w + 1) C) in order, with a segmented scan over the
// owners (a node's positions are contiguous).  A node that lies inside one chunk gets its final bounds here; a node that
// spans chunks leaves one partial per chunk: in head[g] when it began before chunk g, in tail[g] when it begins inside it.
struct BbPart { double mn[3], mx[3]; };

__global__ void __launch_bounds__(kBbThreads) k_bb_bounds(const BbRec *__restrict__ rec, const uint32_t *__restrict__ own, BbNode *__restrict__ nodes,
                                                          uint32_t n, BbPart *__restrict__ head, BbPart *__restrict__ tail) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n_chunks = (n + kBbChunk - 1u) / kBbChunk;
    for (uint32_t g = bb_tid() >> 5; g < n_chunks; g += bb_stride() >> 5) {
        const uint32_t c0 = g * kBbChunk;
        uint32_t carry_o = kBbNone;
        double cmn[3], cmx[3];
        for (uint32_t r = 0; r < kBbChunk / 32u; r++) {
            const uint32_t p = c0 + r * 32u + lane;
            const uint32_t o = p < n ? own[p] : kBbNone;
            double mn[3] = {0, 0, 0}, mx[3] = {0, 0, 0};
            if (o != kBbNone) { const BbRec &x = rec[p]; for (int a = 0; a < 3; a++) { mn[a] = x.mn[a]; mx[a] = x.mx[a]; } }
            for (int off = 1; off < 32; off <<= 1) {                // inclusive segmented scan, the earlier operand first
                const uint32_t o2 = __shfl_up_sync(0xffffffffu, o, off);
                double m2[3], x2[3];
                for (int a = 0; a < 3; a++) { m2[a] = __shfl_up_sync(0xffffffffu, mn[a], off); x2[a] = __shfl_up_sync(0xffffffffu, mx[a], off); }
                if (lane >= (uint32_t)off && o2 == o) for (int a = 0; a < 3; a++) { mn[a] = bb_lo(m2[a], mn[a]); mx[a] = bb_hi(x2[a], mx[a]); }
            }
            if (o != kBbNone && o == carry_o) for (int a = 0; a < 3; a++) { mn[a] = bb_lo(cmn[a], mn[a]); mx[a] = bb_hi(cmx[a], mx[a]); }
            const bool node_ends = o != kBbNone && (p + 1u == n || own[p + 1u] != o);
            const bool chunk_ends = p + 1u == c0 + kBbChunk;
            if (o != kBbNone && (node_ends || chunk_ends)) {
                const uint32_t first = nodes[o].first;
                if (node_ends && first >= c0) {
                    BbNode &nd = nodes[o];
                    for (int a = 0; a < 3; a++) { nd.mn[a] = bb_lo((double)1e30f, mn[a]); nd.mx[a] = bb_hi((double)-1e30f, mx[a]); }
                } else {
                    BbPart &pt = first < c0 ? head[g] : tail[g];
                    for (int a = 0; a < 3; a++) { pt.mn[a] = mn[a]; pt.mx[a] = mx[a]; }
                }
            }
            carry_o = __shfl_sync(0xffffffffu, o, 31);
            for (int a = 0; a < 3; a++) { cmn[a] = __shfl_sync(0xffffffffu, mn[a], 31); cmx[a] = __shfl_sync(0xffffffffu, mx[a], 31); }
        }
    }
}

// the spanning nodes' bounds from their chunk partials, in order; then every node's axis and split plane (bvh.cpp:57-67)
__global__ void __launch_bounds__(kBbThreads) k_bb_finish(BbNode *__restrict__ nodes, uint32_t b, uint32_t e,
                                                          const BbPart *__restrict__ head, const BbPart *__restrict__ tail) {
    for (uint32_t i = b + bb_tid(); i < e; i += bb_stride()) {
        BbNode &nd = nodes[i];
        const uint32_t g0 = nd.first / kBbChunk, g1 = (nd.first + nd.count - 1u) / kBbChunk;
        if (g0 != g1) {
            double mn[3], mx[3];
            for (int a = 0; a < 3; a++) { mn[a] = bb_lo((double)1e30f, tail[g0].mn[a]); mx[a] = bb_hi((double)-1e30f, tail[g0].mx[a]); }
            for (uint32_t g = g0 + 1u; g <= g1; g++)
                for (int a = 0; a < 3; a++) { mn[a] = bb_lo(mn[a], head[g].mn[a]); mx[a] = bb_hi(mx[a], head[g].mx[a]); }
            for (int a = 0; a < 3; a++) { nd.mn[a] = mn[a]; nd.mx[a] = mx[a]; }
        }
        double ext[3];
        for (int a = 0; a < 3; a++) ext[a] = __dsub_rn(nd.mx[a], nd.mn[a]);
        uint32_t axis = 0;
        if (ext[1] > ext[0]) axis = 1;
        if (ext[2] > (double)__double2float_rn(ext[axis])) axis = 2;
        nd.axis = axis;
        nd.split = __fadd_rn(__double2float_rn(nd.mn[axis]), __fmul_rn(__double2float_rn(ext[axis]), 0.5f));
    }
}

// ---- the reference's numbering ------------------------------------------------------------------------------------------
// interior nodes in the subtree of each node of one level (bottom-up, deepest level first)
__global__ void __launch_bounds__(kBbThreads) k_bb_inner(const BbNode *__restrict__ nodes, uint32_t b, uint32_t e, uint32_t *__restrict__ inner) {
    for (uint32_t i = b + bb_tid(); i < e; i += bb_stride()) {
        const uint32_t l = nodes[i].left;
        inner[i] = l ? 1u + inner[l] + inner[l + 1u] : 0u;
    }
}

// top-down: fin[] (final index) and rank[] (interior nodes before it in pre-order) of the children of one level's nodes, and the
// level's nodes written to their final slots
__global__ void __launch_bounds__(kBbThreads) k_bb_number(const BbNode *__restrict__ nodes, uint32_t b, uint32_t e, const uint32_t *__restrict__ inner,
                                                          uint32_t *__restrict__ rank, uint32_t *__restrict__ fin, ct_bvh_node *__restrict__ out) {
    for (uint32_t i = b + bb_tid(); i < e; i += bb_stride()) {
        const BbNode &nd = nodes[i];
        ct_bvh_node o;
        for (int a = 0; a < 3; a++) { o.aabb_min[a] = nd.mn[a]; o.aabb_max[a] = nd.mx[a]; }
        o.first_triangle_index = nd.first;
        o._pad = 0u;
        if (nd.left) {
            const uint32_t l = nd.left, fl = 1u + 2u * rank[i];
            fin[l] = fl; fin[l + 1u] = fl + 1u;
            rank[l] = rank[i] + 1u; rank[l + 1u] = rank[i] + 1u + inner[l];
            o.left_node = fl; o.triangle_count = 0u;
        } else {
            o.left_node = 0u; o.triangle_count = nd.count;
        }
        out[fin[i]] = o;
    }
}

__global__ void __launch_bounds__(kBbThreads) k_bb_indexes(const BbRec *__restrict__ rec, uint32_t n, uint32_t *__restrict__ tri_index) {
    for (uint32_t p = bb_tid(); p < n; p += bb_stride()) tri_index[p] = rec[p].idx;
}

// ---- the whole build ----------------------------------------------------------------------------------------------------
// Every device buffer of one build is carved out of ONE allocation (one cudaMalloc, one cudaFree): sized by a first pass with
// base == nullptr, then carved again from the real allocation.
struct BbArena {
    unsigned char *base = nullptr;
    size_t used = 0;
    template <typename T> T *take(size_t count) {
        const size_t off = (used + 255u) & ~(size_t)255u;
        used = off + std::max<size_t>(count, 1) * sizeof(T);
        return base ? reinterpret_cast<T *>(base + off) : nullptr;
    }
};

struct BbBuffers {
    unsigned char *raw;               // the caller's triangles at their stride
    BbRec *rec[2]; uint32_t *own[2], *S, *NS, *ll_pos, *before, *tile_sum, *inner, *rank, *fin;
    BbNode *nodes; BbPart *head, *tail;
    ct_bvh_node *out;                 // [n_nodes] final numbering
    uint32_t *tri_index;              // [n]
};

void bb_carve(BbArena &a, uint32_t n, size_t raw_bytes, BbBuffers &b) {
    const size_t cap = 2u * (size_t)n - 1u, n_chunks = (n + kBbChunk - 1u) / kBbChunk;
    b.raw = a.take<unsigned char>(raw_bytes);
    b.rec[0] = a.take<BbRec>(n); b.rec[1] = a.take<BbRec>(n);
    b.own[0] = a.take<uint32_t>(n); b.own[1] = a.take<uint32_t>(n);
    b.S = a.take<uint32_t>((size_t)n + 1); b.NS = a.take<uint32_t>((size_t)n + 1);
    b.ll_pos = a.take<uint32_t>(n); b.before = a.take<uint32_t>(n);
    b.tile_sum = a.take<uint32_t>(((size_t)n + 1 + kBbScanTile - 1) / kBbScanTile);
    b.nodes = a.take<BbNode>(cap); b.head = a.take<BbPart>(n_chunks); b.tail = a.take<BbPart>(n_chunks);
    b.inner = a.take<uint32_t>(cap); b.rank = a.take<uint32_t>(cap); b.fin = a.take<uint32_t>(cap);
    b.out = a.take<ct_bvh_node>(cap); b.tri_index = a.take<uint32_t>(n);
}

// Builds the tree over the n triangles in b.raw (at `stride` bytes each) on stream st: b.out[0 .. *n_nodes) and b.tri_index.
// Synchronises once per level.  *depth = levels = the reference's DFS depth.
cudaError_t bb_build(const BbBuffers &bf, uint32_t stride, uint32_t n, int n_sm, cudaStream_t st, uint32_t *n_nodes, int *depth) {
#define BB(call) do { const cudaError_t e_ = (call); if (e_ != cudaSuccess) return e_; } while (0)
    const uint32_t n_chunks = (n + kBbChunk - 1u) / kBbChunk;
    BbRec *const *rec = bf.rec; uint32_t *const *own = bf.own;
    BbNode *nodes = bf.nodes;
    const int grid = n_sm * 8;
    auto blocks_for = [&](uint32_t m) { return (int)std::max<uint32_t>(1u, std::min<uint32_t>((uint32_t)grid, (m + kBbThreads - 1u) / kBbThreads)); };

    k_bb_init<<<blocks_for(n), kBbThreads, 0, st>>>(bf.raw, stride, n, rec[0], own[0], nodes);
    k_bb_bounds<<<blocks_for(n_chunks * 32u), kBbThreads, 0, st>>>(rec[0], own[0], nodes, n, bf.head, bf.tail);
    k_bb_finish<<<1, kBbThreads, 0, st>>>(nodes, 0u, 1u, bf.head, bf.tail);
    BB(cudaGetLastError());
    std::vector<uint32_t> level{0u, 1u};                  // level L = temporary ids [level[L], level[L + 1])
    int cur = 0;
    for (;;) {
        const uint32_t b = level[level.size() - 2], e = level.back(), m = e - b;
        k_bb_pred<<<blocks_for(n + 1u), kBbThreads, 0, st>>>(rec[cur], own[cur], nodes, n, bf.S);
        BB(bb_scan(bf.S, n, bf.tile_sum, st));
        k_bb_nodes<<<blocks_for(m), kBbThreads, 0, st>>>(nodes, b, e, bf.S, bf.before, bf.NS);
        BB(bb_scan(bf.NS, m, bf.tile_sum, st));
        k_bb_children<<<blocks_for(m), kBbThreads, 0, st>>>(nodes, b, e, bf.NS);
        k_bb_pair<<<blocks_for(n), kBbThreads, 0, st>>>(own[cur], nodes, n, bf.S, bf.ll_pos, bf.before);
        k_bb_scatter<<<blocks_for(n), kBbThreads, 0, st>>>(rec[cur], own[cur], nodes, n, bf.S, bf.ll_pos, bf.before, rec[cur ^ 1], own[cur ^ 1]);
        uint32_t splits = 0;
        BB(cudaMemcpyAsync(&splits, bf.NS + m, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        BB(cudaStreamSynchronize(st));
        cur ^= 1;
        if (splits == 0u) break;
        level.push_back(e + 2u * splits);
        k_bb_bounds<<<blocks_for(n_chunks * 32u), kBbThreads, 0, st>>>(rec[cur], own[cur], nodes, n, bf.head, bf.tail);
        k_bb_finish<<<blocks_for(2u * splits), kBbThreads, 0, st>>>(nodes, e, e + 2u * splits, bf.head, bf.tail);
        BB(cudaGetLastError());
    }
    const int levels = (int)level.size() - 1;
    for (int L = levels - 1; L >= 0; L--) k_bb_inner<<<blocks_for(level[L + 1] - level[L]), kBbThreads, 0, st>>>(nodes, level[L], level[L + 1], bf.inner);
    BB(cudaMemsetAsync(bf.rank, 0, sizeof(uint32_t), st));
    BB(cudaMemsetAsync(bf.fin, 0, sizeof(uint32_t), st));
    for (int L = 0; L < levels; L++) k_bb_number<<<blocks_for(level[L + 1] - level[L]), kBbThreads, 0, st>>>(nodes, level[L], level[L + 1], bf.inner, bf.rank, bf.fin, bf.out);
    k_bb_indexes<<<blocks_for(n), kBbThreads, 0, st>>>(rec[cur], n, bf.tri_index);
    BB(cudaGetLastError());
    *n_nodes = level.back();
    *depth = levels;
    return cudaSuccess;
#undef BB
}

}  // namespace
