// ct_build.cuh -- the device-side scene build of ct_gpu_upload_scene (k_build_pairs, k_build_tris).
// Part of the single translation unit ct_gpu.cu (everything lives in its anonymous namespace).
#pragma once

#include "ct_layout.cuh"
#include "ct_bvh_build.cuh"   // bb_scan

namespace {

// ---- scene build on the device (ct_gpu_upload_scene) -------------------------------------------------------------
// The reference's arrays go to the device as they are (nodes, triangles at their stride, the leaf permutation) and
// two kernels turn them into the layout above -- a gather through the permutation plus conversions is bandwidth work
// the host does an order of magnitude slower (868k triangles: 130 ms on 16 host threads, < 1 ms here).  Every value is
// produced by the same IEEE operations as before (fp64 subtractions, round-to-nearest / round-up conversions).
constexpr uint32_t kLeafMark = 0xfffffffeu;       // pid_of[] of a reachable leaf
struct BuildReport {
    unsigned long long bound_bits[3];    // max |bound| over all nodes, per axis (bit pattern of a non-negative double)
    uint32_t boxes_bad;                  // some box is unordered or not finite
    uint32_t bad_pos;                    // a tri_indexes entry out of range (kNoPos: none)
    uint32_t pos0;                       // leaf position of triangle 0
    uint32_t not_nested;                 // some child's box is not inside its parent's box
    uint32_t duplicate;                  // a tri_indexes value occurs twice (with every value in range: not a permutation)
};

// TraceRay recurses unless reflection <= 0 (raythread.cpp:369): a NaN reflection reflects too.  The one test of whether a material
// makes the scene reflective (k_any_reflective).
__device__ __forceinline__ bool reflects(const ct_material &m) { return !(m.reflection <= 0.0f); }

__global__ void __launch_bounds__(256) k_build_pairs(const ct_bvh_node *__restrict__ nodes, const uint32_t *__restrict__ pid_of, uint32_t n_nodes,
                                                     DevPair32 *__restrict__ pairs32, DevPair64 *__restrict__ pairs64,
                                                     uint32_t *__restrict__ pair_parent, uint32_t *__restrict__ tri_parent, uint32_t n_tri, BuildReport *rep) {
    double bound[3] = {0.0, 0.0, 0.0};
    bool bad = false, nest_bad = false;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes; i += gridDim.x * blockDim.x) {
        const ct_bvh_node n = nodes[i];
        const uint32_t pid = pid_of[i];      // interior: its pair; kLeafMark: a leaf; kNoPos: a slot the tree does not reach (may hold anything)
        if (pid == kNoPos) continue;
        for (int a = 0; a < 3; a++) {
            // the filter needs finite, ordered boxes (box_filter picks near/far by the ray's sign)
            if (!(n.aabb_min[a] <= n.aabb_max[a]) || isinf(n.aabb_min[a]) || isinf(n.aabb_max[a])) bad = true;
            else bound[a] = fmax(bound[a], fmax(fabs(n.aabb_min[a]), fabs(n.aabb_max[a])));
        }
        if (n.triangle_count != 0) continue;
        const ct_bvh_node L = nodes[n.left_node], R = nodes[n.left_node + 1u];
        for (int a = 0; a < 3; a++)          // nesting, bit for bit (NaNs fail): what box_maybe's walks rely on
            if (!(L.aabb_min[a] >= n.aabb_min[a] && L.aabb_max[a] <= n.aabb_max[a] && R.aabb_min[a] >= n.aabb_min[a] && R.aabb_max[a] <= n.aabb_max[a])) nest_bad = true;
        DevPair32 p32;
        DevPair64 p64;
        for (int a = 0; a < 3; a++) {
            p64.lmin[a] = L.aabb_min[a]; p64.lmax[a] = L.aabb_max[a]; p64.rmin[a] = R.aabb_min[a]; p64.rmax[a] = R.aabb_max[a];
            p32.lmin[a] = __double2float_rn(L.aabb_min[a]); p32.lmax[a] = __double2float_rn(L.aabb_max[a]);
            p32.rmin[a] = __double2float_rn(R.aabb_min[a]); p32.rmax[a] = __double2float_rn(R.aabb_max[a]);
        }
        p32.l_cnt = L.triangle_count; p32.l_ref = L.triangle_count ? L.first_triangle_index : pid_of[n.left_node];
        p32.r_cnt = R.triangle_count; p32.r_ref = R.triangle_count ? R.first_triangle_index : pid_of[n.left_node + 1u];
        pairs32[pid] = p32;
        pairs64[pid] = p64;
        {
            // who holds whose box: lets candidate_reached find a triangle's leaf box and k_overflow_huge check its ancestor
            // chain without walking down
            for (uint32_t side = 0; side < 2u; side++) {
                const ct_bvh_node &ch = side ? R : L;
                const uint32_t code = 2u * pid + side;
                if (ch.triangle_count == 0) { if (pair_parent) pair_parent[pid_of[n.left_node + side]] = code; }
                else for (uint32_t k = 0; k < ch.triangle_count && (uint64_t)ch.first_triangle_index + k < n_tri; k++) tri_parent[ch.first_triangle_index + k] = code;
            }
        }
    }
    for (int a = 0; a < 3; a++) {
        for (int off = 16; off > 0; off >>= 1) bound[a] = fmax(bound[a], __shfl_xor_sync(0xffffffffu, bound[a], off));
        if ((threadIdx.x & 31u) == 0 && bound[a] > 0.0) atomicMax(&rep->bound_bits[a], (unsigned long long)__double_as_longlong(bound[a]));
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31u) == 0) atomicOr(&rep->boxes_bad, 1u);
    if (__any_sync(0xffffffffu, nest_bad) && (threadIdx.x & 31u) == 0) atomicOr(&rep->not_nested, 1u);
}

__global__ void __launch_bounds__(256) k_build_tris(const unsigned char *__restrict__ raw, uint32_t stride, const uint32_t *__restrict__ tri_indexes,
                                                    uint32_t n_tri, DevTri *__restrict__ tris, DevTri32 *__restrict__ tris32, uint32_t *__restrict__ seen, BuildReport *rep) {
    auto dmax = [](double a, double b) { return (a < b) ? b : a; };      // std::max: a NaN component is skipped
    for (uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x; pos < n_tri; pos += gridDim.x * blockDim.x) {
        const uint32_t k = tri_indexes[pos];
        if (k >= n_tri) { atomicMin(&rep->bad_pos, pos); continue; }
        if (atomicOr(&seen[k >> 5], 1u << (k & 31u)) & (1u << (k & 31u))) { rep->duplicate = 1u; continue; }   // n values in range, none twice: a permutation
        if (k == 0) rep->pos0 = pos;
        const double *v = reinterpret_cast<const double *>(raw + (size_t)k * stride);
        DevTri t;
        DevTri32 t32;
        double k1 = 0.0, k2 = 0.0, k3 = 0.0;
        for (int a = 0; a < 3; a++) {
            t.p1[a] = v[a];
            t.e1[a] = __dsub_rn(v[3 + a], v[a]);
            t.e2[a] = __dsub_rn(v[6 + a], v[a]);
            // fp32 copy + magnitudes for tri_filter_miss (rounded up; NaN k1 = "never certify")
            t32.p1[a] = __double2float_rn(t.p1[a]); t32.e1[a] = __double2float_rn(t.e1[a]); t32.e2[a] = __double2float_rn(t.e2[a]);
            k3 = dmax(k3, fabs(t.p1[a])); k1 = dmax(k1, fabs(t.e1[a])); k2 = dmax(k2, fabs(t.e2[a]));
        }
        t.orig = k; t.pad = 0;
        const bool in_range = k1 >= 0x1p-30 && k1 <= 0x1p30 && k2 >= 0x1p-30 && k2 <= 0x1p30 && k3 <= 0x1p40;   // NaNs fail
        t32.k1 = in_range ? __double2float_ru(k1) : __int_as_float(0x7fc00000);
        t32.k2 = __double2float_ru(k2); t32.k3 = __double2float_ru(k3);
        tris[pos] = t;
        tris32[pos] = t32;
    }
}

// Whether any of n materials reflects (install_scene, whenever the materials are new): *out |= 1.
__global__ void __launch_bounds__(256) k_any_reflective(const ct_material *__restrict__ materials, uint32_t n, uint32_t *out) {
    bool refl = false;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        if (reflects(materials[i])) refl = true;
    if (__any_sync(0xffffffffu, refl) && (threadIdx.x & 31u) == 0) atomicOr(out, 1u);
}

// The one light conversion of ct_gpu_upload_scene and ct_gpu_update_scene: n lights in file order -> DevLight, and the lights that
// cast shadow rays -> DevShadowLight, compacted in file order (the fp32 accumulation of ComputeLighting follows it).  Ambient lights
// cast none (raythread.cpp:284-286); a point light's ray goes to its position (:288), every other type is directional (:293).
// One block of 256 threads: the compaction is a running count, a ballot per warp and the warps' sums per round of 256 lights.
// *n_slights: the shadow lights written.
__global__ void __launch_bounds__(256) k_build_lights(const ct_light *__restrict__ in, uint32_t n, DevLight *__restrict__ lights,
                                                      DevShadowLight *__restrict__ slights, uint32_t *__restrict__ n_slights) {
    __shared__ uint32_t warp_sum[8];
    __shared__ uint32_t base;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (uint32_t first = 0; first < n; first += blockDim.x) {
        const uint32_t i = first + threadIdx.x;
        ct_light L{};
        bool casts = false;
        if (i < n) {
            L = in[i];
            DevLight d;
            d.type = L.type; d.intensity = L.intensity;
            for (int a = 0; a < 3; a++) { d.pos[a] = L.position[a]; d.dir[a] = L.direction[a]; }
            lights[i] = d;
            casts = L.type != CT_LIGHT_AMBIENT;
        }
        const uint32_t ballot = __ballot_sync(0xffffffffu, casts);
        if (lane == 0) warp_sum[warp] = __popc(ballot);
        __syncthreads();
        uint32_t at = base + __popc(ballot & ((1u << lane) - 1u));
        for (uint32_t w = 0; w < warp; w++) at += warp_sum[w];
        if (casts) {
            DevShadowLight sl;
            sl.type = L.type; sl.index = i;
            for (int a = 0; a < 3; a++) sl.v[a] = L.type == CT_LIGHT_POINT ? L.position[a] : L.direction[a];
            slights[at] = sl;
        }
        __syncthreads();
        if (threadIdx.x == 0) for (uint32_t w = 0; w < blockDim.x / 32u; w++) base += warp_sum[w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *n_slights = base;
}

// ---- the early-exit walks' wide tree (DevWide), built from the binary tree on the device --------------------------------
// kWideLevels levels of the reference's tree per wide node, children in DFS order.  Wide nodes are numbered breadth-first: a
// queue, each node's interior children taken in entry order.  One wide level at a time: k_wide_count counts every node's interior
// entries, an exclusive scan over the level's nodes in id order gives their children's ids, k_wide_fill writes the records.  The
// walk starts at the root and follows child links only, so array slots a caller's tree does not reach are never read.
__device__ int wide_entries(const ct_bvh_node *__restrict__ nodes, uint32_t root, uint32_t cur[kWide]) {
    int n_cur = 2;
    cur[0] = nodes[root].left_node; cur[1] = cur[0] + 1u;
    for (int lvl = 1; lvl < kWideLevels; lvl++) {
        uint32_t nxt[kWide];
        int n_nxt = 0;
        for (int i = 0; i < n_cur; i++) {
            const ct_bvh_node &c = nodes[cur[i]];
            if (c.triangle_count != 0) nxt[n_nxt++] = cur[i];
            else { nxt[n_nxt++] = c.left_node; nxt[n_nxt++] = c.left_node + 1u; }
        }
        n_cur = n_nxt;
        for (int i = 0; i < n_cur; i++) cur[i] = nxt[i];
    }
    return n_cur;
}

__global__ void __launch_bounds__(kBbThreads) k_wide_count(const ct_bvh_node *__restrict__ nodes, const uint32_t *__restrict__ root_of,
                                                           uint32_t b, uint32_t e, uint32_t *__restrict__ cnt) {
    for (uint32_t w = b + bb_tid(); w < e; w += bb_stride()) {
        uint32_t cur[kWide];
        const int n_cur = wide_entries(nodes, root_of[w], cur);
        uint32_t c = 0;
        for (int i = 0; i < n_cur; i++) c += nodes[cur[i]].triangle_count == 0 ? 1u : 0u;
        cnt[w - b] = c;
    }
    if (bb_tid() == 0) cnt[e - b] = 0u;
}

__global__ void __launch_bounds__(kBbThreads) k_wide_fill(const ct_bvh_node *__restrict__ nodes, uint32_t *__restrict__ root_of, uint32_t b, uint32_t e,
                                                          const uint32_t *__restrict__ cnt, DevWide *__restrict__ wide) {
    for (uint32_t w = b + bb_tid(); w < e; w += bb_stride()) {
        uint32_t cur[kWide];
        const int n_cur = wide_entries(nodes, root_of[w], cur);
        uint32_t next = e + cnt[w - b];
        DevWide rec;
        for (int i = 0; i < kWide; i++) {
            DevWideChild &x = rec.c[i];
            if (i >= n_cur) {
                for (int a = 0; a < 3; a++) { x.bmin[a] = 1e30f; x.bmax[a] = -1e30f; }
                x.ref = kNoPos; x.cnt = 0u;
                continue;
            }
            const ct_bvh_node &c = nodes[cur[i]];
            for (int a = 0; a < 3; a++) { x.bmin[a] = __double2float_rn(c.aabb_min[a]); x.bmax[a] = __double2float_rn(c.aabb_max[a]); }
            x.cnt = c.triangle_count;
            if (c.triangle_count != 0) x.ref = c.first_triangle_index;
            else { root_of[next] = cur[i]; x.ref = next++; }
        }
        wide[w] = rec;
    }
}

// Collapses the tree below nodes[0] (interior) into wide[0 .. *n_wide); root_of, cnt: scratch of n_pairs + 1 entries, tile_sum of
// (n_pairs + 1) / kBbScanTile + 1.  Synchronises once per wide level.
cudaError_t build_wide(const ct_bvh_node *nodes, uint32_t *root_of, uint32_t *cnt, uint32_t *tile_sum, DevWide *wide, int n_sm,
                       cudaStream_t st, uint32_t *n_wide) {
    const int grid = n_sm * 8;
    auto blocks_for = [&](uint32_t m) { return (int)std::max<uint32_t>(1u, std::min<uint32_t>((uint32_t)grid, (m + kBbThreads - 1u) / kBbThreads)); };
    cudaError_t e = cudaMemsetAsync(root_of, 0, sizeof(uint32_t), st);
    uint32_t b = 0, end = 1;
    while (e == cudaSuccess && b < end) {
        k_wide_count<<<blocks_for(end - b), kBbThreads, 0, st>>>(nodes, root_of, b, end, cnt);
        if ((e = bb_scan(cnt, end - b, tile_sum, st)) != cudaSuccess) break;
        k_wide_fill<<<blocks_for(end - b), kBbThreads, 0, st>>>(nodes, root_of, b, end, cnt, wide);
        uint32_t more = 0;
        if ((e = cudaMemcpyAsync(&more, cnt + (end - b), sizeof more, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) break;
        b = end; end += more;
    }
    *n_wide = end;
    return e;
}

// The interior numbering of a tree built on the device (every node reachable): pid[i] = interior nodes before i, kLeafMark for a
// leaf.  pid holds n_nodes + 1 entries.
__global__ void __launch_bounds__(kBbThreads) k_pid_flags(const ct_bvh_node *__restrict__ nodes, uint32_t n_nodes, uint32_t *__restrict__ pid) {
    for (uint32_t i = bb_tid(); i <= n_nodes; i += bb_stride()) pid[i] = i < n_nodes && nodes[i].triangle_count == 0 ? 1u : 0u;
}
__global__ void __launch_bounds__(kBbThreads) k_pid_leaves(const ct_bvh_node *__restrict__ nodes, uint32_t n_nodes, uint32_t *__restrict__ pid) {
    for (uint32_t i = bb_tid(); i < n_nodes; i += bb_stride()) if (nodes[i].triangle_count != 0) pid[i] = kLeafMark;
}

}  // namespace
