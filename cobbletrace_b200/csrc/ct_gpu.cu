// ct_gpu.cu -- sm_100a wavefront renderer behind the C ABI in include/ct_gpu.h.
//
// Replaces the worker half of the reference's boss/worker (raythread.cpp:437-543
// RayTracePartition -> TraceRay :353 -> ClosestIntersection :197 -> bvh.cpp:198
// IntersectBVHClosest / ComputeLighting :275).  Not a port: the recursive per-pixel CPU loop
// becomes a wavefront of persistent-warp kernels over SoA path state in HBM:
//
//   k_primary   raygen (CanvasToViewport :186) + closest-hit DFS            -> hit records
//   k_emit      the recursion step (:369-373): end the path or append the reflection ray to the next queue
//   k_bounce    the reference's degenerate t=0 reflection rays (:373): first barycentric
//               pass in DFS order (SURVEY 0.4)                               -> hit records
//   k_shadow    ComputeLighting's shadow rays (:288-306), one work item per (light, path) in
//               light-major order (a warp = 32 neighbouring paths, same light); any-hit walk with deferred
//               leaves                                                       -> occlusion bit masks
//   k_shade     NormalOfSceneObject :329 + ComputeLighting :275 accumulation (lights in file
//               order, fp32) + HsvToColor                                    -> per-depth colour stack / framebuffer
//   k_overflow, k_overflow_huge
//               rays whose walk exceeds a visit budget (e.g. shadow rays cast from a shading point
//               4.3e9 units away after a reflection "miss": fp32 slab quotients all round to the
//               same value and EVERY box passes) are parked by k_shadow / k_bounce and finished by a warp
//               each, or -- the every-box-passes ones -- by the whole grid testing all triangles at once
//   k_resolve   unwinds the per-pixel blend chain (:375-379) and stores 0x00BBGGRR pixels
//
// Arithmetic is the reference's mixed fp64/fp32, reproduced exactly: certified fp32 filters decide what they can,
// the reference's own operations (explicit round-to-nearest intrinsics, ct_exact.cuh) decide the rest.
// No tensor cores: the path has no dense contraction.  No CPU fallback.
#include "../../include/ct_gpu.h"
#include "ct_exact.cuh"

#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <cstdlib>
#include <mutex>
#include <string>
#include <thread>
#include <vector>


#include "ct_layout.cuh"     // constants, device structs, Params
#include "ct_traverse.cuh"   // the BVH walks
#include "ct_kernels.cuh"    // the kernels of a tile
#include "ct_bvh_build.cuh"  // the reference's BuildBVH on the device (ct_gpu_build_bvh, CT_FLAG_BUILD_BVH)
#include "ct_build.cuh"      // upload-time scene build kernels

namespace {

// ==== host side of the ABI ===================================================================================
thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorMemoryAllocation ? CT_ERR_OOM : CT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

struct DeviceState {
    bool loaded = false;
    Params p{};
    uint32_t flags = 0;
    bool any_reflective = false;
    int n_sm = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t tile_done[8] = {};   // ring: completion of the last 8 submitted tiles (ct_gpu_throttle)
    unsigned long long tiles_submitted = 0;
    int row_lo = 0, row_hi = 0;      // hull of framebuffer rows rendered since upload (readback clips to it)
    unsigned long long launches = 0; // kernels launched since upload / reset
    cudaEvent_t stage_ev[kMaxLaunches + 1] = {};   // CT_FLAG_STAGE_TIMING: boundaries between the launches of the last tile
    const char *stage_name[kMaxLaunches] = {};
    int stage_depth[kMaxLaunches] = {};
    bool can_overflow = false;       // some traversal could exceed the visit budget: k_overflow launches are needed
    // leaf positions increase along the reference's DFS (bvh_depth).  The parked first-line passes (k_overflow<kFirstLine>,
    // k_overflow_huge) and k_primary_split's replay take the lowest position for the DFS-first one; on a tree without this
    // property reflection rays are never parked and parked primary rays go to k_primary_long (first_line_budget, render_impl)
    bool leaf_dfs_order = true;
    int depth = 0;                   // the tree's depth (the reference's DFS stack entries)
    // per-depth path state (render_impl hands each launch a Params view of its depth, so that the shadow / shade
    // chain of one depth can run on its own stream next to the bounce chain of the next)
    float *hitb_t_all = nullptr; uint32_t *hitb_pos_all = nullptr;      // [depth][cap]
    double *rays_all = nullptr; uint32_t *path_slot_all = nullptr;      // [depth][cap * 6], [depth][cap]
    uint32_t *occ_all = nullptr;                                        // [depth][cap * occ_words]
    uint32_t *parent_q_all = nullptr;                                   // [depth][cap]: parent path of a reflection path (k_emit)
    uint32_t *far_all = nullptr;                                        // [depth][cap]: k_bounce's far lists
    cudaEvent_t ev_lit[16] = {};                                        // shadow verdicts of depth d complete (k_shade of deeper levels may read them)
    unsigned long long rays_shadow_reused = 0;
    OvfRay *ovf_all = nullptr; uint32_t *ovf_huge_all = nullptr;        // [2 * depth + kind][ovf_cap]
    int levels = 1;
    cudaStream_t aux[4] = {};
    cudaEvent_t ev_hit[16] = {}, ev_done[16] = {};
    // multi-GPU frame sharing (ct_gpu_share_*): the cursor and framebuffer a shared render uses (own or the root's)
    unsigned long long *cursor_own = nullptr, *share_cursor = nullptr;
    unsigned long long shared_frames = 0;    // shared renders so far: frame f uses cursor f & 1 (the root zeroes the other one meanwhile)
    int part_index = 0, part_count = 0;      // ct_gpu_share_partition
    bool remote_cursor_ok = true;            // atomics on the attached root's cursor are native (same device, or P2P native atomics)
    uint32_t *share_fb = nullptr;
    void *ipc_opened[2] = {nullptr, nullptr};
    int n_stages = 0;
    bool timed = false;
    // ct_gpu_readback_async: a device-side snapshot of the framebuffer and the stream that copies it to the host
    uint32_t *fb_snapshot = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_snap = nullptr, ev_copied = nullptr;
    bool copy_pending = false;
    void *hot_base = nullptr; size_t hot_bytes = 0;      // pairs32 + tris32 (one allocation): the L2 access-policy window
    size_t l2_window = 0, l2_set_aside = 0;              // what apply_l2_policy obtained (0: none)
    // what the tree's allocations hold (ct_gpu_update_triangles reuses them when the new tree fits): bytes of the hot allocation,
    // pairs64 records, pair_parent entries (its allocation stays when a new tree cannot park: p.pair_parent is then NULL)
    size_t hot_cap = 0;
    uint32_t pairs_cap = 0, pair_parent_cap = 0;
    uint32_t *pair_parent_mem = nullptr;
    std::vector<void *> allocs;
    ct_ray_counters snapshot{};      // totals at the end of the previous counted tile
    unsigned long long rays_overflow = 0, rays_in_place = 0;   // DevTotals' overflow counters as of the last read_totals
    unsigned long long box_exact = 0, tri_exact = 0;
    // rows rendered so far (framebuffer rows), for readback clipping
    int col_lo = 0, col_hi = 0;
};

DeviceState g_dev[kMaxDevices];
std::mutex g_mutex;
// One host thread drives a device at a time (the boss uses one thread per GPU): every entry point that touches a device's
// state holds that device's lock, so a second thread calling in for the same device waits instead of corrupting the state.
std::recursive_mutex g_dev_mutex[kMaxDevices];
#define DEVICE_GUARD(device) std::lock_guard<std::recursive_mutex> dev_lock_(g_dev_mutex[((device) >= 0 && (device) < kMaxDevices) ? (device) : 0])
long long g_budget_option = 0;       // ct_gpu_set_option("traversal_budget"); 0 = default
long long g_warp_budget_option = 0;  // ct_gpu_set_option("overflow_warp_budget"); 0 = default
long long g_any_leaves = 0;               // ct_gpu_set_option("any_leaves"); 0 = by the number of lights
long long g_primary_split = 0;            // ct_gpu_set_option("primary_split"): parked primary rays are finished one ray per warp (k_primary_split)
long long g_primary_budget_option = 0;   // ct_gpu_set_option("primary_budget"); 0 = default (kDefaultPrimaryBudget: never), < 0 = never
long long g_static_eighths = 7;      // ct_gpu_set_option("shared_static_eighths"), see next_chunk
long long g_shared_chunk_shift = 0;  // ct_gpu_set_option("shared_chunk_shift"): 0 = kChunkSharedShift
long long g_run_shift = 0;           // ct_gpu_set_option("shared_run_shift")
long long g_emulate_ranks = 0;       // ct_gpu_set_option("emulate_ranks"): profiling aid, see ct_gpu.h
long long g_shadow_reuse = 1;        // ct_gpu_set_option("shadow_reuse"): a shading point that repeats its parent's takes the parent's shadow verdicts
long long g_hold_frame = 0;          // ct_gpu_set_option("shared_hold_frame"): test aid, see ct_gpu.h
long long g_l2_persist = 1;          // ct_gpu_set_option("l2_persist"): pin the walk's fp32 records in L2 (apply_l2_policy)

int check_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return fail(CT_ERR_NO_DEVICE, "no CUDA device available (%s): this library has no CPU fallback",
                                                 e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    if (device < 0 || device >= n || device >= kMaxDevices) return fail(CT_ERR_NO_DEVICE, "device %d out of range (0..%d)", device, n - 1);
    CU(cudaSetDevice(device));
    return CT_OK;
}

// Hands the persisting L2 lines back and takes the access-policy window off the library's own stream (a caller's stream may be
// gone by now: ct_gpu_set_stream clears it when it is replaced).
void release_l2(DeviceState &s) {
    if (!s.l2_set_aside) return;
    cudaStreamAttrValue attr{};
    attr.accessPolicyWindow.num_bytes = 0;
    if (s.own_stream) cudaStreamSetAttribute(s.own_stream, cudaStreamAttributeAccessPolicyWindow, &attr);
    cudaCtxResetPersistingL2Cache();
    cudaGetLastError();
    s.l2_set_aside = s.l2_window = 0;
}

void free_device(DeviceState &s) {
    release_l2(s);
    for (void *q : s.ipc_opened) if (q) cudaIpcCloseMemHandle(q);
    for (void *p : s.allocs) cudaFree(p);
    s.allocs.clear();
    if (s.ev0) cudaEventDestroy(s.ev0);
    if (s.ev1) cudaEventDestroy(s.ev1);
    for (cudaEvent_t e : s.tile_done) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.stage_ev) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.ev_hit) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.ev_done) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.ev_lit) if (e) cudaEventDestroy(e);
    for (cudaStream_t a : s.aux) if (a) cudaStreamDestroy(a);
    if (s.copy_stream) { cudaStreamSynchronize(s.copy_stream); cudaStreamDestroy(s.copy_stream); }
    if (s.ev_snap) cudaEventDestroy(s.ev_snap);
    if (s.ev_copied) cudaEventDestroy(s.ev_copied);
    if (s.own_stream) cudaStreamDestroy(s.own_stream);
    s = DeviceState{};
}

// The hull of rows holding rendered pixels grows from two sides: tiles this device renders (its own host thread) and rows
// gathered into it from other devices (their host threads, ct_gpu_gather_rows).
std::mutex g_rows_mutex;
void extend_rows(DeviceState &s, int lo, int hi) {
    std::lock_guard<std::mutex> lock(g_rows_mutex);
    if (s.row_hi <= s.row_lo) { s.row_lo = lo; s.row_hi = hi; }
    else { s.row_lo = std::min(s.row_lo, lo); s.row_hi = std::max(s.row_hi, hi); }
}

template <typename T>
int dev_alloc(DeviceState &s, T **out, size_t count, bool zero = false) {
    void *p = nullptr;
    size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) return fail(CT_ERR_OOM, "cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    s.allocs.push_back(p);
    if (zero) CU(cudaMemset(p, 0, bytes));
    *out = static_cast<T *>(p);
    return CT_OK;
}

// frees one allocation of dev_alloc's (cudaFree: waits for the device)
void dev_release(DeviceState &s, void *p) {
    if (!p) return;
    cudaFree(p);
    const auto it = std::find(s.allocs.begin(), s.allocs.end(), p);
    if (it != s.allocs.end()) s.allocs.erase(it);
}

#define TRY(expr) do { int rc_ = (expr); if (rc_ != CT_OK) return rc_; } while (0)


// depth of the reference's DFS (stack entries needed) -- iterative to survive degenerate trees.  Also marks the nodes the
// DFS reaches (array slots nobody points at may hold anything) and rejects leaves whose triangle ranges overlap.  The walk visits
// the nodes in the reference's order (left child, then left + 1) and reports in *dfs_order whether the leaves' triangle ranges
// come in increasing position along it -- true of every tree BuildBVH makes (bvh.cpp:70-97), not of every tree a caller may pass.
int bvh_depth(const ct_bvh_node *nodes, uint32_t n_nodes, uint32_t n_tri, bool *ok, bool *dfs_order, std::vector<uint8_t> &reachable) {
    std::vector<std::pair<uint32_t, int>> st;
    std::vector<uint8_t> covered(n_tri, 0);
    reachable.assign(n_nodes, 0);
    st.push_back({0u, 1});
    int best = 0;
    size_t visited = 0;
    uint64_t next_first = 0;                    // leaf ranges seen so far end below this position
    *ok = true;
    *dfs_order = true;
    while (!st.empty()) {
        auto [i, d] = st.back();
        st.pop_back();
        if (i >= n_nodes || ++visited > (size_t)n_nodes || reachable[i]) { *ok = false; return 0; }      // out of range, a cycle, or a node with two parents
        reachable[i] = 1;
        best = std::max(best, d);
        const ct_bvh_node &nd = nodes[i];
        if (nd.triangle_count == 0) {
            if ((uint64_t)nd.left_node + 1u >= n_nodes || nd.left_node == 0u) { *ok = false; return 0; }
            st.push_back({nd.left_node + 1, d + 1});
            st.push_back({nd.left_node, d + 1});                                  // popped first: the reference's order
        } else {
            if ((uint64_t)nd.first_triangle_index + nd.triangle_count > n_tri) { *ok = false; return 0; }
            if (nd.first_triangle_index < next_first) *dfs_order = false;
            next_first = (uint64_t)nd.first_triangle_index + nd.triangle_count;
            for (uint32_t k = 0; k < nd.triangle_count; k++) {
                uint8_t &c = covered[nd.first_triangle_index + k];
                if (c) { *ok = false; return 0; }                                  // two leaves hold the same position
                c = 1;
            }
        }
    }
    return best;
}

// Device buffers and a stream that live for one ct_gpu_upload_scene or ct_gpu_update_triangles call: the staged copies of the
// caller's arrays, the tree built on the device (arena), the wide tree's scratch.  Freed when the call returns, whatever it returns.
// async: the buffers come from the stream-ordered allocator and are freed in st's order (cudaFree would wait for the whole device;
// the update's arena is allocated on the caller's stream, which st has waited for).
struct Staging {
    std::vector<void *> ptrs;
    BbArena arena;
    cudaStream_t st = nullptr;
    bool async = false;
    cudaEvent_t ready = nullptr;
    ~Staging() {
        if (async) {
            if (arena.base) cudaFreeAsync(arena.base, st);
            for (void *q : ptrs) cudaFreeAsync(q, st);
        }
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
        if (ready) cudaEventDestroy(ready);
        if (!async) { cudaFree(arena.base); for (void *q : ptrs) cudaFree(q); }
    }
    template <typename T> cudaError_t alloc(T **out, size_t count) {
        void *q = nullptr;
        const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
        const cudaError_t e = async ? cudaMallocAsync(&q, bytes, st) : cudaMalloc(&q, bytes);
        if (e == cudaSuccess) ptrs.push_back(q);
        *out = static_cast<T *>(q);
        return e;
    }
};

// ---- the scene built from a tree: one builder for ct_gpu_upload_scene and ct_gpu_update_triangles ------------------------------
// A binary tree in the reference's layout on the device and what the scene arrays are made from with it.
struct DeviceTree {
    const ct_bvh_node *nodes = nullptr;
    const uint32_t *pid = nullptr;           // interior numbering: pair of an interior node, kLeafMark for a leaf, kNoPos unreachable
    const uint32_t *tri_index = nullptr;
    const unsigned char *tris = nullptr;     // the triangles at `stride`
    uint32_t stride = 72, n_nodes = 0, n_pairs = 0;
    ct_bvh_node root{};
    int depth = 0;
    DevWide *wide = nullptr;                 // the early-exit walks' wide tree, in scratch (collapse_wide)
    uint32_t n_wide = 0;
};

// The reference's BuildBVH over the n triangles in bf.raw on stg.st (bb_build), then the interior numbering k_build_pairs takes
// (k_pid_flags, bb_scan, k_pid_leaves).  Synchronises stg.st once per level.  A tree deeper than the device traversal stack is
// CT_ERR_LIMIT, before anything else is allocated.
int build_device_tree(Staging &stg, const BbBuffers &bf, uint32_t stride, uint32_t n, int n_sm, DeviceTree &t) {
    CU(bb_build(bf, stride, n, n_sm, stg.st, &t.n_nodes, &t.depth));
    CU(cudaMemcpyAsync(&t.root, bf.out, sizeof t.root, cudaMemcpyDeviceToHost, stg.st));
    CU(cudaStreamSynchronize(stg.st));
    if (t.depth > kStackMax) return fail(CT_ERR_LIMIT, "BVH depth %d exceeds the device traversal stack (%d)", t.depth, kStackMax);
    t.n_pairs = (t.n_nodes - 1u) / 2u;                                      // every node is reachable: 1 + 2 * interior nodes
    uint32_t *pid = nullptr, *ptile = nullptr;                              // interior numbering: a scan over the node order
    CU(stg.alloc(&pid, (size_t)t.n_nodes + 1)); CU(stg.alloc(&ptile, ((size_t)t.n_nodes + 1) / kBbScanTile + 1));
    const int blocks = std::max(1, std::min(n_sm * 8, (int)((t.n_nodes + kBbThreads) / kBbThreads)));
    k_pid_flags<<<blocks, kBbThreads, 0, stg.st>>>(bf.out, t.n_nodes, pid);
    CU(bb_scan(pid, t.n_nodes, ptile, stg.st));
    k_pid_leaves<<<blocks, kBbThreads, 0, stg.st>>>(bf.out, t.n_nodes, pid);
    CU(cudaGetLastError());
    t.nodes = bf.out; t.pid = pid; t.tri_index = bf.tri_index; t.tris = bf.raw; t.stride = stride;
    return CT_OK;
}

// The early-exit walks' wide tree into scratch (none for a leaf root).  Synchronises stg.st.
int collapse_wide(Staging &stg, DeviceTree &t, int n_sm) {
    if (t.root.triangle_count == 0) {
        uint32_t *root_of = nullptr, *wcnt = nullptr, *wtile = nullptr;
        CU(stg.alloc(&t.wide, t.n_pairs)); CU(stg.alloc(&root_of, (size_t)t.n_pairs + 1)); CU(stg.alloc(&wcnt, (size_t)t.n_pairs + 1));
        CU(stg.alloc(&wtile, ((size_t)t.n_pairs + 1) / kBbScanTile + 1));
        CU(build_wide(t.nodes, root_of, wcnt, wtile, t.wide, n_sm, stg.st, &t.n_wide));
    }
    CU(cudaStreamSynchronize(stg.st));
    return CT_OK;
}

// The records every walk step reads -- the wide tree, fp32 child pairs and fp32 triangles -- share ONE allocation, so that a single
// L2 access-policy window can cover them (apply_l2_policy): wide at 0, pairs32 at pairs_at, tris32 at tris_at.
struct HotLayout { size_t pairs_at, tris_at, bytes; };
HotLayout hot_layout(uint32_t n_wide, uint32_t n_pairs, uint32_t n_tri) {
    const size_t pair_bytes = ((size_t)std::max<uint32_t>(n_pairs, 1) * sizeof(DevPair32) + 255u) & ~(size_t)255u;
    const size_t wide_bytes = ((size_t)n_wide * sizeof(DevWide) + 255u) & ~(size_t)255u;
    return {wide_bytes, wide_bytes + pair_bytes, wide_bytes + pair_bytes + (size_t)n_tri * sizeof(DevTri32)};
}

// Parked rays: only when a DFS can run past the visit budget at all.
bool walks_can_park(const Params &p, uint32_t n_nodes) { return (uint64_t)n_nodes + p.n_tri > p.budget; }

// Parked rays per launch: 2^18 (16 MB) -- with primary walks parked as well (option "primary_budget": 2-3 % of a dragon-class
// frame's primary rays) 1/16 of the frame's paths where that is more; a full buffer means finishing rays in place, which must
// stay hypothetical.
uint32_t parking_cap(const Params &p) { return p.primary_budget > 0u ? std::max<uint32_t>(1u << 18, p.cap / 16u) : 1u << 18; }

// Where the scene arrays go.  pair_parent may be NULL (no walk can be parked).
struct SceneArrays { unsigned char *hot; DevPair64 *pairs64; uint32_t *pair_parent, *tri_parent; DevTri *tris; };

// The scene arrays from tree t (k_build_pairs, k_build_tris, the wide tree copied into the hot allocation at hot_layout's offsets)
// and what the build reports about them.  materials: the scene's, by original id, already on the device.  The scratch is taken
// before anything is written; the rest is enqueued on st, which is synchronised.
int build_scene_arrays(Staging &stg, cudaStream_t st, const DeviceTree &t, const ct_material *materials, uint32_t n_tri, const SceneArrays &out,
                       int n_sm, BuildReport *rep) {
    uint32_t *seen = nullptr; BuildReport *drep = nullptr;
    const size_t seen_words = ((size_t)n_tri + 31u) / 32u;
    CU(stg.alloc(&drep, 1));
    CU(stg.alloc(&seen, seen_words));
    const HotLayout hl = hot_layout(t.n_wide, t.n_pairs, n_tri);
    DevPair32 *dp32 = reinterpret_cast<DevPair32 *>(out.hot + hl.pairs_at);
    DevTri32 *dt32 = reinterpret_cast<DevTri32 *>(out.hot + hl.tris_at);
    if (t.n_wide) CU(cudaMemcpyAsync(out.hot, t.wide, (size_t)t.n_wide * sizeof(DevWide), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemsetAsync(seen, 0, seen_words * 4, st));
    *rep = BuildReport{};
    rep->bad_pos = kNoPos; rep->pos0 = kNoPos;
    CU(cudaMemcpyAsync(drep, rep, sizeof *rep, cudaMemcpyHostToDevice, st));
    if (out.pair_parent) CU(cudaMemsetAsync(out.pair_parent, 0xff, (size_t)std::max<uint32_t>(t.n_pairs, 1) * 4, st));
    CU(cudaMemsetAsync(out.tri_parent, 0xff, (size_t)n_tri * 4, st));
    const int build_blocks = n_sm * 8;
    k_build_pairs<<<build_blocks, 256, 0, st>>>(t.nodes, t.pid, t.n_nodes, dp32, out.pairs64, out.pair_parent, out.tri_parent, n_tri, drep);
    k_build_tris<<<build_blocks, 256, 0, st>>>(t.tris, t.stride, t.tri_index, materials, n_tri, out.tris, dt32, seen, drep);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(rep, drep, sizeof *rep, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return CT_OK;
}

// What the frame kernels read about the tree, from t and its build report; pointers into out as build_scene_arrays wrote them.
void set_tree(DeviceState &s, const DeviceTree &t, const SceneArrays &out, const BuildReport &rep) {
    Params &p = s.p;
    const HotLayout hl = hot_layout(t.n_wide, t.n_pairs, p.n_tri);
    p.root_cnt = t.root.triangle_count;
    p.root_ref = t.root.triangle_count ? t.root.first_triangle_index : 0u;      // an interior root is pair 0
    p.n_pairs = t.n_pairs;
    p.n_nodes = t.n_nodes;
    p.wide = t.n_wide ? reinterpret_cast<const DevWide *>(out.hot) : nullptr;
    p.n_wide = t.n_wide;
    p.pos_of_tri0 = rep.pos0;
    p.nested = (!rep.not_nested && !rep.boxes_bad) ? 1u : 0u;
    for (int a = 0; a < 3; a++) {
        double bound;
        memcpy(&bound, &rep.bound_bits[a], sizeof bound);
        p.bound[a] = (!rep.boxes_bad && bound < 1e30) ? bound : INFINITY;
        p.root_min[a] = t.root.aabb_min[a]; p.root_max[a] = t.root.aabb_max[a];
        p.root_min32[a] = (float)p.root_min[a]; p.root_max32[a] = (float)p.root_max[a];
    }
    p.pairs32 = reinterpret_cast<const DevPair32 *>(out.hot + hl.pairs_at); p.pairs64 = out.pairs64;
    p.tris = out.tris; p.tris32 = reinterpret_cast<const DevTri32 *>(out.hot + hl.tris_at);
    p.pair_parent = out.pair_parent; p.tri_parent = out.tri_parent;
    s.hot_base = out.hot; s.hot_bytes = hl.bytes;
    s.depth = t.depth;
}

int launch_grid(const DeviceState &s, int blocks_per_sm) { return s.n_sm * blocks_per_sm; }

// The walk budget of the first-line (reflection) rays: unlimited -- never parked, the walk in the ray's own thread keeps the
// reference's DFS order on any tree -- when leaf positions do not increase along the DFS (DeviceState::leaf_dfs_order).  The cost
// on such a tree: a reflection ray cast from a shading point 2^32 ray lengths away walks the whole tree in one thread.
uint32_t first_line_budget(const DeviceState &s) { return s.leaf_dfs_order ? s.p.budget : 0xffffffffu; }

// The primary rays k_primary parked into v.ovf (slot 0 of the parking buffers) are finished by k_primary_split (option
// "primary_split", one ray per warp) or by k_primary_long (32 to a warp).  k_primary_split's replay takes leaf positions for the
// reference's test order, so a tree whose leaf positions do not increase along the DFS (DeviceState::leaf_dfs_order) always gets
// k_primary_long.  Returns true when k_primary_split was launched.
bool launch_parked_primary(const DeviceState &s, const Params &v, bool count, cudaStream_t st, int work_idx) {
    if (g_primary_split && s.leaf_dfs_order) {
        if (count) k_primary_split<true><<<s.n_sm * 4, kOvfThreads, 0, st>>>(v);
        else k_primary_split<false><<<s.n_sm * 4, kOvfThreads, 0, st>>>(v);
        return true;
    }
    if (count) k_primary_long<true><<<launch_grid(s, 8), kBlockThreads, 0, st>>>(v, work_idx);
    else k_primary_long<false><<<launch_grid(s, 8), kBlockThreads, 0, st>>>(v, work_idx);
    return false;
}

// L2 residency of the walk's hot set.  The fp32 child pairs and fp32 triangles (76 MB for the dragon-class scene) are
// read by every walk step, at random; everything else a frame touches (ray queues, hit records, occlusion masks, colour
// stacks, the fp64 records behind the filters) streams through once.  Left to the default policy the streams evict the
// tree (measured: 70 % L2 hit rate on a hot set that fits, every other warp step waiting for DRAM).  So: set aside as
// much L2 as the device allows for persisting lines and open an access-policy window over the hot allocation on every
// stream the tile's kernels run on; hitRatio scales the window down to the set-aside size when the scene is larger.
int apply_l2_policy(DeviceState &s, int device, cudaStream_t st) {
    if (!g_l2_persist || !s.hot_base || s.hot_bytes == 0) return CT_OK;
    int persisting_max = 0, window_max = 0;           // (two attributes: cudaGetDeviceProperties takes milliseconds)
    CU(cudaDeviceGetAttribute(&persisting_max, cudaDevAttrMaxPersistingL2CacheSize, device));
    CU(cudaDeviceGetAttribute(&window_max, cudaDevAttrMaxAccessPolicyWindowSize, device));
    if (persisting_max <= 0 || window_max <= 0) return CT_OK;
    if (s.l2_set_aside == 0) {
        const size_t want = std::min<size_t>(s.hot_bytes, (size_t)persisting_max);
        if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) != cudaSuccess) { cudaGetLastError(); return CT_OK; }
        size_t got = 0;
        cudaDeviceGetLimit(&got, cudaLimitPersistingL2CacheSize);
        s.l2_set_aside = got;
        s.l2_window = std::min<size_t>(s.hot_bytes, (size_t)window_max);
    }
    if (s.l2_set_aside == 0) return CT_OK;
    cudaStreamAttrValue attr{};
    attr.accessPolicyWindow.base_ptr = s.hot_base;
    attr.accessPolicyWindow.num_bytes = s.l2_window;
    attr.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)s.l2_set_aside / (double)s.l2_window);
    attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(st, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
    return CT_OK;
}

int read_totals(DeviceState &s, ct_ray_counters *out) {   // synchronises the stream
    DevTotals h;
    CU(cudaMemcpyAsync(&h, s.p.tot, sizeof h, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    out->rays_primary = h.rays_primary; out->rays_shadow = h.rays_shadow; out->rays_reflection = h.rays_reflection;
    out->box_tests = h.box_tests; out->tri_tests = h.tri_tests;
    s.rays_overflow = h.rays_overflow; s.rays_in_place = h.rays_in_place;
    s.box_exact = h.box_exact; s.tri_exact = h.tri_exact;
    s.rays_shadow_reused = h.rays_shadow_reused;
    return CT_OK;
}

// The one path of the ray queries (ct_gpu_trace_rays) and of the KAT entries ct_gpu_debug_early / ct_gpu_debug_primary: n rays in
// device memory of one kind, the walk of the frame's kernel for that kind with this call's scratch as its hit records, occlusion
// words and parking buffers, the real second-pass kernels for the parked rays, then k_ray_results.  Enqueued on `st`; the scratch
// is one stream-ordered allocation, freed in stream order.
// park_cap: the primary rays' parking buffer, 0 = a frame's.  path (may be NULL): how each ray was finished (ct_gpu_debug_*).
int trace_impl(DeviceState &s, int kind, uint32_t n, const double *org, const double *dir, uint32_t *found, uint32_t *index,
               float *tclosest, uint32_t *path, uint32_t park_cap, cudaStream_t st) {
    const bool primary = kind == CT_RAY_PRIMARY;
    const bool park = primary ? s.can_overflow && s.p.primary_budget > 0u : s.can_overflow;      // render_impl's rules
    uint32_t ovf_cap = 0;
    if (park) ovf_cap = std::min<uint32_t>(n, primary && park_cap ? std::min(park_cap, s.p.ovf_cap) : s.p.ovf_cap);
    // the scratch: scheduler and totals records, one occlusion word and one hit record per ray, the parking buffer and huge list --
    // carved from one allocation (first pass: sizes only)
    char *base = nullptr;
    size_t used = 0;
    auto take = [&](size_t bytes) { char *q = base ? base + used : nullptr; used += (bytes + 255u) & ~(size_t)255u; return q; };
    DevSched *sched = nullptr; DevTotals *tot = nullptr; uint32_t *occ = nullptr, *hpos = nullptr, *huge = nullptr; float *ht = nullptr;
    OvfRay *ovf = nullptr;
    auto carve = [&]() {
        used = 0;
        sched = (DevSched *)take(sizeof(DevSched)); tot = (DevTotals *)take(sizeof(DevTotals));
        occ = (uint32_t *)take(4ull * n); ht = (float *)take(4ull * n); hpos = (uint32_t *)take(4ull * n);
        if (ovf_cap) { ovf = (OvfRay *)take(sizeof(OvfRay) * (size_t)ovf_cap); huge = (uint32_t *)take(4ull * ovf_cap); }
    };
    carve();
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&base), used, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? CT_ERR_OOM : CT_ERR_CUDA, "cudaMallocAsync(%zu bytes): %s", used, cudaGetErrorString(e));
    }
    carve();
    Params v = s.p;
    v.sched = sched; v.tot = tot; v.occ = occ; v.occ_words = 1;
    v.hit0_t = v.hitb_t = ht; v.hit0_pos = v.hitb_pos = hpos;
    v.cap = n; v.max_depth = 0; v.dbg_found = nullptr; v.dbg_index = nullptr; v.dbg_t = nullptr;
    v.ovf = ovf; v.ovf_huge = huge; v.ovf_cap = ovf_cap; v.split_path = path;
    if (kind == CT_RAY_REFLECTION) v.budget = first_line_budget(s);
    // everything below is enqueued; a failure still frees the scratch in stream order
    auto enqueue = [&]() -> cudaError_t {
        cudaError_t r = cudaMemsetAsync(sched, 0, (size_t)((char *)occ - (char *)sched), st);       // DevSched and DevTotals
        if (r != cudaSuccess) return r;
        const uint32_t blocks = (n + kBlockThreads - 1) / kBlockThreads;
        if (primary) {
            if (park) k_debug_primary<true><<<blocks, kBlockThreads, 0, st>>>(v, n, org, dir, path);
            else k_debug_primary<false><<<blocks, kBlockThreads, 0, st>>>(v, n, org, dir, path);
            if (park) launch_parked_primary(s, v, false, st, 0);
        } else if (kind == CT_RAY_SHADOW) {
            k_debug_early<kAnyHit><<<blocks, kBlockThreads, 0, st>>>(v, n, org, dir, path);
            if (park) { k_overflow<kAnyHit, false><<<s.n_sm * 2, kOvfThreads, 0, st>>>(v, 0); k_overflow_huge<kAnyHit, false><<<s.n_sm * 4, 256, 0, st>>>(v, 0); }
        } else {
            k_debug_early<kFirstLine><<<blocks, kBlockThreads, 0, st>>>(v, n, org, dir, path);
            if (park) { k_overflow<kFirstLine, false><<<s.n_sm * 2, kOvfThreads, 0, st>>>(v, 0); k_overflow_huge<kFirstLine, false><<<s.n_sm * 4, 256, 0, st>>>(v, 0); }
        }
        const int mode = primary ? kClosest : kind == CT_RAY_SHADOW ? kAnyHit : kFirstLine;
        k_ray_results<<<(n + 255) / 256, 256, 0, st>>>(v, mode, n, found, index, tclosest, path);
        return cudaGetLastError();
    };
    const cudaError_t r = enqueue();
    const cudaError_t f = cudaFreeAsync(base, st);
    if (r != cudaSuccess) return fail(CT_ERR_CUDA, "ray query: %s", cudaGetErrorString(r));
    if (f != cudaSuccess) return fail(CT_ERR_CUDA, "cudaFreeAsync: %s", cudaGetErrorString(f));
    return CT_OK;
}

// ct_gpu_debug_early / ct_gpu_debug_primary: host arrays in and out around trace_impl on the render stream, rays in the caller's
// order (each ray's path code is that of the ray-by-ray tested walk), synchronous.
int debug_query(int device, int kind, uint32_t n, const double *origins, const double *directions, uint32_t park_cap,
                uint32_t *found, uint32_t *index, float *tclosest, uint32_t *path) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (n == 0) return CT_OK;
    double *d_o = nullptr, *d_d = nullptr; uint32_t *d_f = nullptr, *d_i = nullptr, *d_p = nullptr; float *d_tc = nullptr;
    int rc = CT_OK;
    auto cleanup = [&]() { cudaFree(d_o); cudaFree(d_d); cudaFree(d_f); cudaFree(d_i); cudaFree(d_p); cudaFree(d_tc); };
#define CUX(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(CT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); cleanup(); return rc; } } while (0)
    CUX(cudaMalloc(&d_o, 24ull * n)); CUX(cudaMalloc(&d_d, 24ull * n));
    CUX(cudaMalloc(&d_f, 4ull * n)); CUX(cudaMalloc(&d_i, 4ull * n)); CUX(cudaMalloc(&d_p, 4ull * n)); CUX(cudaMalloc(&d_tc, 4ull * n));
    CUX(cudaMemcpy(d_o, origins, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_d, directions, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaStreamSynchronize(s.stream));
    rc = trace_impl(s, kind, n, d_o, d_d, d_f, d_i, kind == CT_RAY_SHADOW ? nullptr : d_tc, d_p, park_cap, s.stream);
    if (rc != CT_OK) { cudaStreamSynchronize(s.stream); cleanup(); return rc; }
    CUX(cudaStreamSynchronize(s.stream));
    if (found) CUX(cudaMemcpy(found, d_f, 4ull * n, cudaMemcpyDeviceToHost));
    if (index) CUX(cudaMemcpy(index, d_i, 4ull * n, cudaMemcpyDeviceToHost));
    if (tclosest) CUX(cudaMemcpy(tclosest, d_tc, 4ull * n, cudaMemcpyDeviceToHost));
    if (path) CUX(cudaMemcpy(path, d_p, 4ull * n, cudaMemcpyDeviceToHost));
    cleanup();
#undef CUX
    return CT_OK;
}

// The per-depth path state the stages of a tile or of a shade query batch work on: [depth][cap] arrays as DeviceState describes
// them, parking buffers [2 * depth + kind][ovf_cap].  A frame's are allocated at upload, a query's per call (shade_impl).
struct PathArrays {
    float *hitb_t_all; uint32_t *hitb_pos_all;
    double *rays_all; uint32_t *path_slot_all;
    uint32_t *occ_all, *parent_q_all, *far_all;
    OvfRay *ovf_all; uint32_t *ovf_huge_all;
};

// The stages of one tile (render_impl) or of one batch of a shade query (shade_impl, QUERY: the query forms of k_primary, k_shadow,
// k_shade and k_resolve).  pk: what every launch starts from, pk.max_depth the depth the recursion goes to (0 without a reflective
// material).  serial: every launch on st in the order written (CT_FLAG_STAGE_TIMING, and queries); otherwise each depth's lighting
// chain runs on a side stream of its own (s.aux, DESIGN.md 4).  mark(name, depth) is called after each stage enqueued on st (side
// stream stages: in serial mode only); `launches` counts the rest.
template <bool QUERY, class Mark>
int enqueue_stages(DeviceState &s, const Params &pk, const PathArrays &a, bool count, bool serial, cudaStream_t st, Mark &&mark,
                   unsigned long long &launches) {
    const int depth_max = pk.max_depth;
    const int grid = launch_grid(s, 8);
    int work = 0;
    // Params as the launches of depth d see them: their own hit records, occlusion masks, ray queue in / out
    auto view = [&](int d) {
        Params v = pk;
        const size_t cap = pk.cap;
        if (a.hitb_t_all) { v.hitb_t = a.hitb_t_all + cap * d; v.hitb_pos = a.hitb_pos_all + cap * d; }
        if (a.rays_all) {
            v.ray_buf[d & 1] = a.rays_all + cap * 6 * d;            v.path_slot[d & 1] = a.path_slot_all + cap * d;
            v.ray_buf[(d & 1) ^ 1] = a.rays_all + cap * 6 * (d + 1); v.path_slot[(d & 1) ^ 1] = a.path_slot_all + cap * (d + 1);
            v.parent_q[d & 1] = a.parent_q_all + cap * d; v.parent_q[(d & 1) ^ 1] = a.parent_q_all + cap * (d + 1);
        }
        v.occ = a.occ_all + cap * pk.occ_words * d;
        if (a.far_all) v.far_list = a.far_all + cap * d;
        return v;
    };
    auto overflow = [&](const Params &v0, cudaStream_t q, int mode_anyhit, int ovf_idx, int depth) -> int {   // parked rays of the launch just made
        if (!s.can_overflow) return CT_OK;
        Params v = v0;
        v.ovf = a.ovf_all + (size_t)pk.ovf_cap * ovf_idx; v.ovf_huge = a.ovf_huge_all + (size_t)pk.ovf_cap * ovf_idx;
        const int g1 = s.n_sm * 2, g2 = s.n_sm * 4;
        if (mode_anyhit) {
            if (count) { k_overflow<kAnyHit, true><<<g1, kOvfThreads, 0, q>>>(v, ovf_idx); k_overflow_huge<kAnyHit, true><<<g2, 256, 0, q>>>(v, ovf_idx); }
            else { k_overflow<kAnyHit, false><<<g1, kOvfThreads, 0, q>>>(v, ovf_idx); k_overflow_huge<kAnyHit, false><<<g2, 256, 0, q>>>(v, ovf_idx); }
        } else {
            if (count) { k_overflow<kFirstLine, true><<<g1, kOvfThreads, 0, q>>>(v, ovf_idx); k_overflow_huge<kFirstLine, true><<<g2, 256, 0, q>>>(v, ovf_idx); }
            else { k_overflow<kFirstLine, false><<<g1, kOvfThreads, 0, q>>>(v, ovf_idx); k_overflow_huge<kFirstLine, false><<<g2, 256, 0, q>>>(v, ovf_idx); }
        }
        launches++;                                         // two kernels, one stage
        return mark(mode_anyhit ? "overflow_shadow" : "overflow_bounce", depth);
    };
    // Two dependency chains per frame (DESIGN.md 4):
    //   hits      primary -> emit(0) -> bounce(1) -> emit(1) -> bounce(2) -> ...          (main stream)
    //   lighting  shadow(d) -> shade(d), needs only the hits of depth d                   (one side stream per depth)
    // so the lighting of depth d overlaps the hit chain of depth d+1 and the lighting of the other depths; the
    // persistent CTAs of a later kernel move into an SM as those of an earlier one run out of work, which fills
    // the kernels' tails.  Serial: everything on the main stream instead.
    // (Queries never count tests: count is false for them, and the query forms have no COUNT instantiations.)
    {
        Params v0 = view(0);              // (k_primary also runs the recursion step of depth 0: it needs the depth's queues)
        // walks longer than primary_budget pair visits are parked (slot 0 of the parking buffers: depth 0 has no bounce launch)
        // and walked again by k_primary_long, in warps made of long walks only
        const bool park_primary = s.can_overflow && pk.primary_budget > 0u;
        v0.ovf = park_primary ? a.ovf_all : nullptr;
        if (park_primary) {
            if (count) { if constexpr (!QUERY) k_primary<true, true><<<grid, kBlockThreads, 0, st>>>(v0); }
            else k_primary<false, true, QUERY><<<grid, kBlockThreads, 0, st>>>(v0);
        } else {
            if (count) { if constexpr (!QUERY) k_primary<true, false><<<grid, kBlockThreads, 0, st>>>(v0); }
            else k_primary<false, false, QUERY><<<grid, kBlockThreads, 0, st>>>(v0);
        }
        TRY(mark("primary", 0));
        if (park_primary) {
            const bool split = launch_parked_primary(s, v0, count, st, work);
            if (!split) work++;
            TRY(mark(split ? "primary_split" : "primary_long", 0));
        }
    }
    for (int d = 0; d <= depth_max; d++) {
        const Params v = view(d);
        const int ovf_b = 2 * d, ovf_s = 2 * d + 1;
        if (d > 0) {
            Params vb = v;
            vb.budget = first_line_budget(s);
            if (s.can_overflow) { vb.ovf = a.ovf_all + (size_t)pk.ovf_cap * ovf_b; vb.ovf_huge = a.ovf_huge_all + (size_t)pk.ovf_cap * ovf_b; }
            if (count) k_bounce<true><<<grid, kBlockThreads, 0, st>>>(vb, d, work++, ovf_b);
            else k_bounce<false><<<grid, kBlockThreads, 0, st>>>(vb, d, work++, ovf_b);
            TRY(mark("bounce", d));
            TRY(overflow(v, st, 0, ovf_b, d));
        }
        cudaStream_t side = serial ? st : s.aux[d % 4];
        if (!serial) { CU(cudaEventRecord(s.ev_hit[d], st)); CU(cudaStreamWaitEvent(side, s.ev_hit[d], 0)); }
        if (depth_max > 0) {
            // TraceRay's recursion step runs inside the hit kernels (emit_paths); what is left for a kernel of its own are the
            // reflection paths k_bounce had parked, whose hit k_overflow has just delivered
            if (d > 0 && s.can_overflow) {
                k_emit<<<s.n_sm * 2, kBlockThreads, 0, st>>>(v, d, work++, a.ovf_all + (size_t)pk.ovf_cap * ovf_b, ovf_b);
                TRY(mark("emit_late", d));
            }
        }
        if (pk.n_slights > 0) {
            Params vs = v;
            if (s.can_overflow) { vs.ovf = a.ovf_all + (size_t)pk.ovf_cap * ovf_s; vs.ovf_huge = a.ovf_huge_all + (size_t)pk.ovf_cap * ovf_s; }
            if (count) { if constexpr (!QUERY) k_shadow<true><<<grid, kBlockThreads, 0, side>>>(vs, d, work++, ovf_s); }
            else k_shadow<false, QUERY><<<grid, kBlockThreads, 0, side>>>(vs, d, work++, ovf_s);
            if (serial) TRY(mark("shadow", d)); else launches++;
            if (serial) { TRY(overflow(v, side, 1, ovf_s, d)); }
            else if (s.can_overflow) {
                Params vo = v;
                vo.ovf = a.ovf_all + (size_t)pk.ovf_cap * ovf_s; vo.ovf_huge = a.ovf_huge_all + (size_t)pk.ovf_cap * ovf_s;
                if (count) { k_overflow<kAnyHit, true><<<s.n_sm * 2, kOvfThreads, 0, side>>>(vo, ovf_s); k_overflow_huge<kAnyHit, true><<<s.n_sm * 4, 256, 0, side>>>(vo, ovf_s); }
                else { k_overflow<kAnyHit, false><<<s.n_sm * 2, kOvfThreads, 0, side>>>(vo, ovf_s); k_overflow_huge<kAnyHit, false><<<s.n_sm * 4, 256, 0, side>>>(vo, ovf_s); }
                launches += 2;
            }
        }
        if (!serial) {
            // k_shade(d) may read the shadow verdicts of shallower depths (occlusion_source): they are complete at ev_lit
            CU(cudaEventRecord(s.ev_lit[d], side));
            for (int dd = 0; dd < d; dd++) CU(cudaStreamWaitEvent(side, s.ev_lit[dd], 0));
        }
        k_shade<QUERY><<<grid, kBlockThreads, 0, side>>>(v, d, work++);
        if (serial) TRY(mark("shade", d)); else launches++;
        if (!serial) CU(cudaEventRecord(s.ev_done[d], side));
    }
    if (!serial) for (int d = 0; d <= depth_max; d++) CU(cudaStreamWaitEvent(st, s.ev_done[d], 0));
    if (depth_max > 0) { k_resolve<QUERY><<<s.n_sm * 4, 256, 0, st>>>(pk); TRY(mark("resolve", 0)); }
    if (pk.supersample) { k_supersample<<<s.n_sm * 4, 256, 0, st>>>(pk); TRY(mark("supersample", 0)); }
    if (pk.subsample) { k_subsample<<<s.n_sm * 4, 256, 0, st>>>(pk); TRY(mark("subsample", 0)); }
    return CT_OK;
}


// Rays a shade query takes per batch: its path state is carved for this many, whatever n is (the bound ct_gpu.h states).
constexpr uint32_t kShadeBatch = 1u << 20;

// ct_gpu_shade_rays: TraceRay (raythread.cpp:353-386) for n caller rays, recursion depth max_depth, through the frame's own stages
// (enqueue_stages<true>, serialised on st) -- the caller's ray i is depth-0 slot i of its batch, its colour goes to color[i].  The
// batches of at most kShadeBatch rays reuse one stream-ordered allocation: the path state of every level, carved like upload's, and
// parking buffers of min(batch, the frame's ovf_cap) rays.  Nothing is synchronised; the scratch is freed in stream order.
int shade_impl(DeviceState &s, uint32_t n, int max_depth, const double *org, const double *dir, uint32_t *color, cudaStream_t st) {
    const int depth_max = s.any_reflective ? max_depth : 0;       // render_impl's rule: without a reflective material TraceRay stops at :369
    const size_t levels = (size_t)depth_max + 1;
    const uint32_t batch = std::min(n, kShadeBatch);
    const size_t cap = (batch + kChunkMax - 1u) / kChunkMax * kChunkMax;
    const uint32_t ovf_cap = s.can_overflow ? std::min<uint32_t>(batch, s.p.ovf_cap) : 0u;
    const size_t words = s.p.occ_words;
    char *base = nullptr;
    size_t used = 0;
    auto take = [&](size_t bytes) { char *q = base ? base + used : nullptr; used += (bytes + 255u) & ~(size_t)255u; return q; };
    Params pk = s.p;
    PathArrays a{};
    auto carve = [&]() {                                            // (first pass: sizes only)
        used = 0;
        pk.sched = (DevSched *)take(sizeof(DevSched)); pk.tot = (DevTotals *)take(sizeof(DevTotals));
        pk.hit0_t = (float *)take(4 * cap); pk.hit0_pos = (uint32_t *)take(4 * cap);
        pk.stack_color = (uint32_t *)take(4 * cap * levels);
        pk.term_level = (uint8_t *)take(cap);
        pk.own_chunks = (uint32_t *)take(4 * ((cap >> kChunkLocalShift) + 1));
        a.occ_all = (uint32_t *)take(4 * cap * words * levels);
        if (ovf_cap) { a.ovf_all = (OvfRay *)take(sizeof(OvfRay) * ovf_cap * 2 * levels); a.ovf_huge_all = (uint32_t *)take(4ull * ovf_cap * 2 * levels); }
        if (levels > 1) {
            a.hitb_t_all = (float *)take(4 * cap * levels); a.hitb_pos_all = (uint32_t *)take(4 * cap * levels);
            pk.stack_refl = (float *)take(4 * cap * levels);
            a.rays_all = (double *)take(48 * cap * (levels + 1)); a.path_slot_all = (uint32_t *)take(4 * cap * (levels + 1));
            a.parent_q_all = (uint32_t *)take(4 * cap * (levels + 1));
            a.far_all = (uint32_t *)take(4 * cap * levels);
        }
    };
    carve();
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&base), used, st);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? CT_ERR_OOM : CT_ERR_CUDA, "cudaMallocAsync(%zu bytes): %s", used, cudaGetErrorString(e));
    }
    carve();
    if (levels == 1) pk.stack_refl = nullptr;
    pk.max_depth = depth_max;
    pk.cap = (uint32_t)cap;
    pk.occ = a.occ_all;
    pk.parent_q_all = a.parent_q_all; pk.hitb_t_all = a.hitb_t_all; pk.occ_all = a.occ_all;
    pk.reuse_shadow = (g_shadow_reuse && a.parent_q_all) ? 1u : 0u;
    pk.ovf = a.ovf_all; pk.ovf_huge = a.ovf_huge_all; pk.ovf_cap = ovf_cap;
    // one device, its own cursor, chunks of 32 rays: what render_impl sets up for a tile rendered alone, without emulate_ranks
    pk.steal = &pk.sched->steal_local;
    pk.chunk_shift = kChunkLocalShift; pk.steal_stride = 1u; pk.part_index = pk.part_count = 0u; pk.run_shift = 0u;
    pk.fb = pk.fb_out = nullptr; pk.dbg_found = pk.dbg_index = nullptr; pk.dbg_t = nullptr; pk.split_path = nullptr;
    pk.subsample = pk.supersample = 0;
    unsigned long long launches = 0;                                // (not the device's: queries leave ct_gpu_kernel_launches alone)
    int rc = CT_OK;
    cudaError_t r = cudaMemsetAsync(pk.tot, 0, sizeof(DevTotals), st);
    for (uint32_t first = 0; r == cudaSuccess && rc == CT_OK && first < n; first += batch) {
        Params v = pk;
        v.n_slots = std::min(batch, n - first);
        v.q_org = org + 3ull * first; v.q_dir = dir + 3ull * first;
        v.final_color = color + first;
        if ((r = cudaMemsetAsync(pk.sched, 0, sizeof(DevSched), st)) != cudaSuccess) break;
        rc = enqueue_stages<true>(s, v, a, false, true, st, [](const char *, int) { return (int)CT_OK; }, launches);
    }
    if (r == cudaSuccess) r = cudaGetLastError();
    const cudaError_t f = cudaFreeAsync(base, st);
    if (rc != CT_OK) return rc;
    if (r != cudaSuccess) return fail(CT_ERR_CUDA, "shade query: %s", cudaGetErrorString(r));
    if (f != cudaSuccess) return fail(CT_ERR_CUDA, "cudaFreeAsync: %s", cudaGetErrorString(f));
    return CT_OK;
}

// A query's array: device (or managed) memory of `device`, aligned.  Checked before anything is enqueued.
int check_device_array(int device, const void *p, size_t align, const char *name) {
    if ((uintptr_t)p % align) return fail(CT_ERR_INVALID, "%s is not %zu-byte aligned", name, align);
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return fail(CT_ERR_INVALID, "%s: not a CUDA pointer", name); }
    if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != device)
        return fail(CT_ERR_INVALID, "%s is not device memory of device %d", name, device);
    return CT_OK;
}
}  // namespace

// ==== exported C ABI ==========================================================================================
extern "C" {

int ct_gpu_abi_version(void) { return CT_GPU_ABI_VERSION; }

const char *ct_gpu_last_error(void) { return g_err; }

int ct_gpu_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(CT_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    return n;
}

int ct_gpu_upload_scene(int device, const ct_scene_desc *d) {
    if (!d || d->struct_size != sizeof(ct_scene_desc)) return fail(CT_ERR_INVALID, "ct_scene_desc missing or struct_size != %zu", sizeof(ct_scene_desc));
    if (d->n_triangles == 0 || !d->triangles || !d->materials) return fail(CT_ERR_INVALID, "scene has no triangles");
    if (d->triangle_stride < 72 || d->triangle_stride % 8) return fail(CT_ERR_INVALID, "triangle_stride must be >= 72 and a multiple of 8");
    const bool build = (d->flags & CT_FLAG_BUILD_BVH) != 0;
    if (build) {
        if (d->n_nodes != 0 || d->nodes || d->tri_indexes) return fail(CT_ERR_INVALID, "CT_FLAG_BUILD_BVH builds the tree: n_nodes must be 0, nodes and tri_indexes NULL");
        if (d->n_triangles >= (1u << 31)) return fail(CT_ERR_LIMIT, "%u triangles: the device build takes fewer than 2^31", d->n_triangles);
    } else if (d->n_nodes == 0 || !d->nodes || !d->tri_indexes) {
        return fail(CT_ERR_INVALID, "scene has no BVH (build it with the reference's BuildBVH or ct_host_build_bvh, or pass CT_FLAG_BUILD_BVH)");
    }
    if (d->n_lights && !d->lights) return fail(CT_ERR_INVALID, "n_lights > 0 but lights == NULL");
    if (d->width <= 0 || d->height <= 0 || (int64_t)d->width * d->height > (1ll << 30)) return fail(CT_ERR_INVALID, "bad frame size %dx%d", d->width, d->height);
    if (d->max_depth < 0 || d->max_depth > 15) return fail(CT_ERR_LIMIT, "max_depth %d outside 0..15", d->max_depth);
    if ((d->flags & CT_FLAG_SUPERSAMPLING) && (d->flags & CT_FLAG_KEEP_HITS))
        return fail(CT_ERR_INVALID, "CT_FLAG_SUPERSAMPLING cannot be combined with CT_FLAG_KEEP_HITS (a pixel has 16 primary rays)");
    bool ok = true, dfs_order = true;          // a tree BuildBVH makes has its leaves in DFS order (bvh.cpp:70-97)
    std::vector<uint8_t> reachable;
    int depth = 0;
    if (!build) {
        depth = bvh_depth(d->nodes, d->n_nodes, d->n_triangles, &ok, &dfs_order, reachable);
        if (!ok) return fail(CT_ERR_INVALID, "BVH is malformed (child or triangle range out of bounds, overlapping leaves, a cycle or a shared child)");
        if (depth > kStackMax) return fail(CT_ERR_LIMIT, "BVH depth %d exceeds the device traversal stack (%d)", depth, kStackMax);
    }
    TRY(check_device(device));
    DEVICE_GUARD(device);
    std::lock_guard<std::mutex> lock(g_mutex);
    DeviceState &s = g_dev[device];
    const bool timing = getenv("CT_GPU_TIMING") != nullptr;
    auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double t_begin = now_ms();
    double t_mark = t_begin;
    auto lap = [&](const char *what) { if (timing) { double t = now_ms(); fprintf(stderr, "ct_gpu_upload_scene: %-28s %7.1f ms\n", what, t - t_mark); t_mark = t; } };
    int n_sm = 0;
    CU(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));

    // The binary tree, the leaf permutation and the triangles on the device.  With CT_FLAG_BUILD_BVH the tree is built here, into
    // buffers of the upload's own, BEFORE the previous scene is released: a refused tree leaves that scene loaded.
    const size_t tri_bytes = (size_t)(d->n_triangles - 1) * d->triangle_stride + 72;      // the last triangle may end at its third vertex
    Staging stg;
    CU(cudaStreamCreateWithFlags(&stg.st, cudaStreamNonBlocking));
    DeviceTree t;
    if (build) {
        BbBuffers bf;
        bb_carve(stg.arena, d->n_triangles, tri_bytes, bf);
        CU(cudaMalloc(&stg.arena.base, stg.arena.used));
        stg.arena.used = 0;
        bb_carve(stg.arena, d->n_triangles, tri_bytes, bf);
        CU(cudaMemcpyAsync(bf.raw, d->triangles, tri_bytes, cudaMemcpyHostToDevice, stg.st));
        TRY(build_device_tree(stg, bf, d->triangle_stride, d->n_triangles, n_sm, t));
        lap("BVH built on the device");
    } else {
        t.root = d->nodes[0];
        t.n_nodes = d->n_nodes; t.depth = depth; t.stride = d->triangle_stride;
        // nodes: reference layout -> per-interior-node child pairs, built on the device from the raw arrays (k_build_pairs); the host
        // only numbers the interior nodes it validated
        std::vector<uint32_t> pid_of(d->n_nodes, kNoPos);
        for (uint32_t i = 0; i < d->n_nodes; i++)
            if (reachable[i]) pid_of[i] = d->nodes[i].triangle_count == 0 ? t.n_pairs++ : kLeafMark;      // unreachable slots get no record and write nothing
        ct_bvh_node *rn = nullptr; uint32_t *rp = nullptr, *ri = nullptr; unsigned char *rt = nullptr;
        CU(stg.alloc(&rn, d->n_nodes)); CU(stg.alloc(&rp, d->n_nodes)); CU(stg.alloc(&ri, d->n_triangles)); CU(stg.alloc(&rt, tri_bytes));
        CU(cudaMemcpyAsync(rn, d->nodes, (size_t)d->n_nodes * sizeof(ct_bvh_node), cudaMemcpyHostToDevice, stg.st));
        CU(cudaMemcpyAsync(rp, pid_of.data(), (size_t)d->n_nodes * 4, cudaMemcpyHostToDevice, stg.st));
        CU(cudaMemcpyAsync(ri, d->tri_indexes, (size_t)d->n_triangles * 4, cudaMemcpyHostToDevice, stg.st));
        CU(cudaMemcpyAsync(rt, d->triangles, tri_bytes, cudaMemcpyHostToDevice, stg.st));
        t.nodes = rn; t.pid = rp; t.tri_index = ri; t.tris = rt;
        lap("interior-node numbering (host)");
    }
    // the early-exit walks' wide tree, into scratch first: its size decides the layout of the hot allocation below
    TRY(collapse_wide(stg, t, n_sm));
    lap("wide tree (device)");

    free_device(s);
    s.n_sm = n_sm;
    CU(cudaStreamCreateWithFlags(&s.own_stream, cudaStreamNonBlocking));
    s.stream = s.own_stream;
    CU(cudaEventCreate(&s.ev0));
    CU(cudaEventCreate(&s.ev1));
    for (cudaEvent_t &e : s.tile_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaEvent_t &e : s.ev_hit) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaEvent_t &e : s.ev_done) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaEvent_t &e : s.ev_lit) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (cudaStream_t &a : s.aux) CU(cudaStreamCreateWithFlags(&a, cudaStreamNonBlocking));
    if (d->flags & CT_FLAG_STAGE_TIMING) for (cudaEvent_t &e : s.stage_ev) CU(cudaEventCreate(&e));
    s.p.budget = g_budget_option > 0 ? (uint32_t)std::min<long long>(g_budget_option, 1ll << 30) : kDefaultBudget;
    s.p.warp_budget = g_warp_budget_option > 0 ? (uint32_t)std::min<long long>(g_warp_budget_option, 1ll << 30) : kWarpBudget;
    s.p.primary_budget = g_primary_budget_option < 0 ? 0u : g_primary_budget_option > 0 ? (uint32_t)std::min<long long>(g_primary_budget_option, 1ll << 30) : kDefaultPrimaryBudget;
    s.flags = d->flags;
    s.leaf_dfs_order = dfs_order;

    Params &p = s.p;
    p.n_tri = d->n_triangles; p.n_lights = d->n_lights;
    s.can_overflow = walks_can_park(p, t.n_nodes);

    SceneArrays out{};
    ct_material *dm = nullptr;
    const uint32_t pairs = std::max<uint32_t>(t.n_pairs, 1);
    s.hot_cap = hot_layout(t.n_wide, t.n_pairs, d->n_triangles).bytes;
    TRY(dev_alloc(s, &out.hot, s.hot_cap));
    TRY(dev_alloc(s, &out.pairs64, pairs)); s.pairs_cap = pairs;
    TRY(dev_alloc(s, &out.tris, d->n_triangles)); TRY(dev_alloc(s, &dm, d->n_triangles));
    TRY(dev_alloc(s, &out.tri_parent, d->n_triangles));
    if (s.can_overflow) { TRY(dev_alloc(s, &out.pair_parent, pairs)); s.pair_parent_mem = out.pair_parent; s.pair_parent_cap = pairs; }
    BuildReport rep{};
    {
        const cudaError_t e = cudaMemcpyAsync(dm, d->materials, (size_t)d->n_triangles * sizeof(ct_material), cudaMemcpyHostToDevice, s.stream);
        if (e != cudaSuccess) { free_device(s); CU(e); }
        const int rc = build_scene_arrays(stg, s.stream, t, dm, d->n_triangles, out, s.n_sm, &rep);
        if (rc != CT_OK) { free_device(s); return rc; }
    }
    if (rep.bad_pos != kNoPos) { free_device(s); return fail(CT_ERR_INVALID, "tri_indexes[%u] = %u out of range", rep.bad_pos, build ? 0u : d->tri_indexes[rep.bad_pos]); }
    if (rep.duplicate || rep.pos0 == kNoPos) { free_device(s); return fail(CT_ERR_INVALID, "tri_indexes is not a permutation of 0..n_triangles-1 (an index occurs twice)"); }
    s.any_reflective = rep.any_reflective != 0;
    set_tree(s, t, out, rep);
    p.materials = dm;
    lap("scene arrays built on the device");
    std::vector<DevLight> lights(std::max<uint32_t>(d->n_lights, 1));
    for (uint32_t i = 0; i < d->n_lights; i++) {
        lights[i].type = d->lights[i].type; lights[i].intensity = d->lights[i].intensity;
        for (int a = 0; a < 3; a++) { lights[i].pos[a] = d->lights[i].position[a]; lights[i].dir[a] = d->lights[i].direction[a]; }
    }
    std::vector<DevShadowLight> slights;
    for (uint32_t i = 0; i < d->n_lights; i++) {
        if (d->lights[i].type == CT_LIGHT_AMBIENT) continue;            // raythread.cpp:284-286: no shadow ray
        DevShadowLight sl{};
        sl.type = d->lights[i].type; sl.index = i;
        const double *v = (sl.type == CT_LIGHT_POINT) ? d->lights[i].position : d->lights[i].direction;   // :288 / :293 (every non-point light is directional)
        for (int a = 0; a < 3; a++) sl.v[a] = v[a];
        slights.push_back(sl);
    }
    p.n_slights = (uint32_t)slights.size();
    // the any-hit walk's leaf-list length trades the lit rays' phase overhead against the occluded rays' early exit: measured 12 best for
    // the 3-light dragon frame (k_shadow 1.11 ms against 1.15 at 8), 8 for the 66-light scene (6.75 ms against 7.14 at 12) -- a shading point
    // inside a sphere of lights has half of them behind its own surface.  Option "any_leaves" overrides (0 = this rule).
    p.any_leaves = g_any_leaves > 0 ? (uint32_t)g_any_leaves : (p.n_slights >= 16u ? 8u : 12u);
    p.occ_words = std::max<uint32_t>((d->n_lights + 31u) / 32u, 1u);
    DevLight *dl = nullptr; DevShadowLight *dsl = nullptr;
    TRY(dev_alloc(s, &dl, lights.size()));
    TRY(dev_alloc(s, &dsl, slights.size()));
    if (!slights.empty()) CU(cudaMemcpy(dsl, slights.data(), slights.size() * sizeof(DevShadowLight), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dl, lights.data(), lights.size() * sizeof(DevLight), cudaMemcpyHostToDevice));
    p.slights = dsl; p.lights = dl;

    memcpy(p.cam, d->camera_position, sizeof p.cam);
    memcpy(p.rot, d->camera_rotation, sizeof p.rot);
    p.vp_w = d->viewport[0]; p.vp_h = d->viewport[1]; p.vp_d = d->viewport[2];
    p.W = d->width; p.H = d->height; p.max_depth = d->max_depth; p.background = d->background;

    // x range: the reference's centred square (raythread.cpp:454-455) or the whole width
    int half = d->height / 2;
    int x_lo = -half, n_x = 2 * half;
    if (d->flags & CT_FLAG_WIDE) { x_lo = -(d->width / 2); n_x = d->width; }
    p.x_lo = x_lo; p.n_x = n_x;
    p.blocks_x = (n_x + 7) / 8;
    s.col_lo = std::max(0, x_lo + d->width / 2);
    s.col_hi = std::min(d->width, x_lo + n_x + d->width / 2);
    int rows_max = 2 * half + 1;
    {
        const uint64_t pixel_slots = (uint64_t)p.blocks_x * (uint64_t)((rows_max + 3) / 4) * 32u;
        const uint64_t slots = pixel_slots * ((d->flags & CT_FLAG_SUPERSAMPLING) ? 16u : 1u);
        if (slots > (1ull << 31)) { free_device(s); return fail(CT_ERR_LIMIT, "frame needs %llu path slots (limit 2^31)", (unsigned long long)slots); }
        p.cap = (uint32_t)((slots + kChunkMax - 1u) / kChunkMax * kChunkMax);
    }

    const int levels = s.any_reflective ? d->max_depth + 1 : 1;
    TRY(dev_alloc(s, &p.hit0_t, p.cap)); TRY(dev_alloc(s, &p.hit0_pos, p.cap));
    TRY(dev_alloc(s, &p.stack_color, (size_t)p.cap * levels));
    TRY(dev_alloc(s, &p.term_level, p.cap, true));
    s.levels = levels;
    TRY(dev_alloc(s, &s.occ_all, (size_t)p.cap * p.occ_words * levels, true));
    p.occ = s.occ_all;
    if (s.can_overflow) {
        p.ovf_cap = parking_cap(p);
        TRY(dev_alloc(s, &s.ovf_all, (size_t)p.ovf_cap * 2 * levels));
        TRY(dev_alloc(s, &s.ovf_huge_all, (size_t)p.ovf_cap * 2 * levels));
        p.ovf = s.ovf_all; p.ovf_huge = s.ovf_huge_all;
    }
    if (levels > 1) {
        TRY(dev_alloc(s, &s.hitb_t_all, (size_t)p.cap * levels)); TRY(dev_alloc(s, &s.hitb_pos_all, (size_t)p.cap * levels));
        TRY(dev_alloc(s, &p.stack_refl, (size_t)p.cap * levels));
        TRY(dev_alloc(s, &s.rays_all, (size_t)p.cap * 6 * (levels + 1))); TRY(dev_alloc(s, &s.path_slot_all, (size_t)p.cap * (levels + 1)));
        TRY(dev_alloc(s, &s.parent_q_all, (size_t)p.cap * (levels + 1)));
        TRY(dev_alloc(s, &s.far_all, (size_t)p.cap * levels));
    }
    TRY(dev_alloc(s, &p.fb, (size_t)d->width * d->height, true));       // calloc'd like cobbletrace.cpp:57
    p.subsample = (d->flags & CT_FLAG_SUBSAMPLING) ? 1 : 0;
    p.supersample = (d->flags & CT_FLAG_SUPERSAMPLING) ? 1 : 0;
    if (p.subsample || p.supersample) TRY(dev_alloc(s, &p.final_color, p.cap, true));
    TRY(dev_alloc(s, &p.own_chunks, (p.cap >> kChunkLocalShift) + 1u));
    TRY(dev_alloc(s, &s.cursor_own, 2 * kCursorStride, true));           // its own allocation: exported over CUDA IPC; two cursors, 128 bytes apart
    s.share_cursor = s.cursor_own; s.share_fb = p.fb;
    if (d->flags & CT_FLAG_KEEP_HITS) {
        size_t npx = (size_t)d->width * d->height;
        TRY(dev_alloc(s, &p.dbg_found, npx)); TRY(dev_alloc(s, &p.dbg_index, npx, true)); TRY(dev_alloc(s, &p.dbg_t, npx, true));
        CU(cudaMemset(p.dbg_found, 0xff, npx * sizeof(uint32_t)));
    }
    TRY(dev_alloc(s, &p.sched, 1, true));
    TRY(dev_alloc(s, &p.tot, 1, true));
    lap("path state allocation");
    TRY(apply_l2_policy(s, device, s.stream));
    for (cudaStream_t a : s.aux) TRY(apply_l2_policy(s, device, a));
    if (timing) fprintf(stderr, "ct_gpu_upload_scene: L2 window %zu bytes, set-aside %zu bytes; total %.1f ms\n", s.l2_window, s.l2_set_aside, now_ms() - t_begin);
    s.loaded = true;
    return CT_OK;
}

int ct_gpu_build_bvh(int device, uint32_t n_triangles, const void *triangles, uint32_t triangle_stride, ct_bvh_node *nodes,
                     uint32_t nodes_capacity, uint32_t *tri_indexes) {
    if (n_triangles == 0) return fail(CT_ERR_INVALID, "cannot build a BVH over zero triangles");
    if (n_triangles >= (1u << 31)) return fail(CT_ERR_LIMIT, "%u triangles: the device build takes fewer than 2^31", n_triangles);
    if (!triangles || !nodes || !tri_indexes) return fail(CT_ERR_INVALID, "triangles, nodes and tri_indexes must not be NULL");
    if (triangle_stride < 72 || triangle_stride % 8) return fail(CT_ERR_INVALID, "triangle_stride must be >= 72 and a multiple of 8");
    if (nodes_capacity < 2u * n_triangles - 1u) return fail(CT_ERR_INVALID, "nodes_capacity %u < 2 n - 1 = %u", nodes_capacity, 2u * n_triangles - 1u);
    TRY(check_device(device));
    DEVICE_GUARD(device);
    auto cu_fail = [](cudaError_t e, const char *what) {
        return fail(e == cudaErrorMemoryAllocation ? CT_ERR_OOM : CT_ERR_CUDA, "ct_gpu_build_bvh: %s: %s", what, cudaGetErrorString(e));
    };
    int n_sm = 0;
    cudaError_t e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return cu_fail(e, "cudaDeviceGetAttribute");
    // a stream and buffers of its own: a scene uploaded on this device is not touched
    const bool timing = getenv("CT_GPU_TIMING") != nullptr;
    auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    double t_mark = now_ms();
    auto lap = [&](const char *what) { if (timing) { double t = now_ms(); fprintf(stderr, "ct_gpu_build_bvh: %-28s %7.2f ms\n", what, t - t_mark); t_mark = t; } };
    cudaStream_t st = nullptr;
    if ((e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)) != cudaSuccess) return cu_fail(e, "cudaStreamCreate");
    BbArena arena;
    struct Release { cudaStream_t s; BbArena &a; ~Release() { cudaStreamSynchronize(s); cudaStreamDestroy(s); cudaFree(a.base); } } release{st, arena};
    const size_t tri_bytes = (size_t)(n_triangles - 1) * triangle_stride + 72;      // the last triangle may end at its third vertex
    BbBuffers bf;
    bb_carve(arena, n_triangles, tri_bytes, bf);
    if ((e = cudaMalloc(&arena.base, arena.used)) != cudaSuccess) { arena.base = nullptr; return cu_fail(e, "cudaMalloc"); }
    arena.used = 0;
    bb_carve(arena, n_triangles, tri_bytes, bf);
    lap("allocation");
    if ((e = cudaMemcpyAsync(bf.raw, triangles, tri_bytes, cudaMemcpyHostToDevice, st)) != cudaSuccess) return cu_fail(e, "cudaMemcpyAsync");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cu_fail(e, "cudaStreamSynchronize");
    lap("triangles to the device");
    uint32_t n_nodes = 0;
    int depth = 0;
    if ((e = bb_build(bf, triangle_stride, n_triangles, n_sm, st, &n_nodes, &depth)) != cudaSuccess) return cu_fail(e, "build");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cu_fail(e, "cudaStreamSynchronize");
    if (timing) fprintf(stderr, "ct_gpu_build_bvh: %u nodes, %d levels\n", n_nodes, depth);
    lap("tree built on the device");
    if (n_nodes > (uint32_t)INT32_MAX) return fail(CT_ERR_LIMIT, "%u nodes do not fit the return value", n_nodes);
    if ((e = cudaMemcpyAsync(nodes, bf.out, (size_t)n_nodes * sizeof(ct_bvh_node), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return cu_fail(e, "cudaMemcpyAsync");
    if ((e = cudaMemcpyAsync(tri_indexes, bf.tri_index, (size_t)n_triangles * sizeof(uint32_t), cudaMemcpyDeviceToHost, st)) != cudaSuccess) return cu_fail(e, "cudaMemcpyAsync");
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return cu_fail(e, "cudaStreamSynchronize");
    lap("tree to the host");
    return (int)n_nodes;
}

// The scene ct_gpu_upload_scene with CT_FLAG_BUILD_BVH would load from the caller's triangles and the loaded scene's materials,
// lights, camera and frame, built by the same functions into the loaded scene's arrays: the tree in scratch first (a refused or
// failed build changes nothing), then -- after the device has finished the work in flight -- the scene arrays over the live ones.
// Everything else the device holds stays.
int ct_gpu_update_triangles(int device, const ct_triangle_update *u) {
    if (!u || u->struct_size != sizeof(ct_triangle_update)) return fail(CT_ERR_INVALID, "ct_triangle_update missing or struct_size != %zu", sizeof(ct_triangle_update));
    if (!u->triangles) return fail(CT_ERR_INVALID, "NULL triangles");
    if (u->triangle_stride < 72 || u->triangle_stride % 8) return fail(CT_ERR_INVALID, "triangle_stride must be >= 72 and a multiple of 8");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    std::lock_guard<std::mutex> lock(g_mutex);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    Params &p = s.p;
    if (u->n_triangles != p.n_tri) return fail(CT_ERR_INVALID, "%u triangles: the loaded scene has %u (a re-upload changes the count)", u->n_triangles, p.n_tri);
    TRY(check_device_array(device, u->triangles, 8, "triangles"));
    const bool timing = getenv("CT_GPU_TIMING") != nullptr;
    auto now_ms = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; };
    const double t_begin = now_ms();
    double t_mark = t_begin;
    auto lap = [&](const char *what) { if (timing) { double t = now_ms(); fprintf(stderr, "ct_gpu_update_triangles: %-28s %7.2f ms\n", what, t - t_mark); t_mark = t; } };
    const cudaStream_t st = u->stream ? static_cast<cudaStream_t>(u->stream) : s.stream;
    const uint32_t n = p.n_tri;
    const size_t tri_bytes = (size_t)(n - 1) * u->triangle_stride + 72;      // the last triangle may end at its third vertex

    // the caller's triangles into the build's arena in `st`'s order; the build runs on the scratch stream behind them
    Staging stg;
    stg.async = true;
    CU(cudaStreamCreateWithFlags(&stg.st, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&stg.ready, cudaEventDisableTiming));
    BbBuffers bf;
    bb_carve(stg.arena, n, tri_bytes, bf);
    {
        const cudaError_t e = cudaMallocAsync(reinterpret_cast<void **>(&stg.arena.base), stg.arena.used, st);
        if (e != cudaSuccess) { cudaGetLastError(); stg.arena.base = nullptr; CU(e); }
    }
    stg.arena.used = 0;
    bb_carve(stg.arena, n, tri_bytes, bf);
    {
        const cudaError_t c = cudaMemcpyAsync(bf.raw, u->triangles, tri_bytes, cudaMemcpyDeviceToDevice, st);
        cudaError_t w = cudaEventRecord(stg.ready, st);
        if (w == cudaSuccess) w = cudaStreamWaitEvent(stg.st, stg.ready, 0);
        if (w != cudaSuccess) cudaStreamSynchronize(st);              // the arena is freed in stg.st's order: after the copy
        CU(c); CU(w);
    }
    DeviceTree t;
    TRY(build_device_tree(stg, bf, u->triangle_stride, n, s.n_sm, t));
    lap("BVH built on the device");
    TRY(collapse_wide(stg, t, s.n_sm));
    lap("wide tree (device)");

    // The live allocations the new tree needs: the hot allocation, pairs64 and pair_parent are reused where the new records fit,
    // the parking buffers appear when walks can be parked for the first time.  New ones are taken before anything is written.
    const HotLayout hl = hot_layout(t.n_wide, t.n_pairs, n);
    const uint32_t pairs = std::max<uint32_t>(t.n_pairs, 1);
    const bool can_overflow = walks_can_park(p, t.n_nodes);
    SceneArrays out{};
    out.hot = hl.bytes <= s.hot_cap ? static_cast<unsigned char *>(s.hot_base) : nullptr;
    out.pairs64 = pairs <= s.pairs_cap ? const_cast<DevPair64 *>(p.pairs64) : nullptr;
    out.pair_parent = !can_overflow ? nullptr : pairs <= s.pair_parent_cap ? s.pair_parent_mem : nullptr;
    out.tri_parent = const_cast<uint32_t *>(p.tri_parent);
    out.tris = const_cast<DevTri *>(p.tris);
    const bool new_hot = !out.hot, new_pairs = !out.pairs64, new_parent = can_overflow && !out.pair_parent, new_parking = can_overflow && !s.ovf_all;
    OvfRay *ovf = nullptr; uint32_t *ovf_huge = nullptr;
    const uint32_t ovf_cap = new_parking ? parking_cap(p) : p.ovf_cap;
    auto take = [&]() -> int {
        if (new_hot) TRY(dev_alloc(s, &out.hot, hl.bytes));
        if (new_pairs) TRY(dev_alloc(s, &out.pairs64, pairs));
        if (new_parent) TRY(dev_alloc(s, &out.pair_parent, pairs));
        if (new_parking) { TRY(dev_alloc(s, &ovf, (size_t)ovf_cap * 2 * s.levels)); TRY(dev_alloc(s, &ovf_huge, (size_t)ovf_cap * 2 * s.levels)); }
        return CT_OK;
    };
    auto give_back = [&]() {                                         // the new allocations of a call that fails
        if (new_hot) dev_release(s, out.hot);
        if (new_pairs) dev_release(s, out.pairs64);
        if (new_parent) dev_release(s, out.pair_parent);
        dev_release(s, ovf); dev_release(s, ovf_huge);
    };
    int rc = take();
    if (rc != CT_OK) { give_back(); return rc; }
    lap("allocation");

    // frames and queries in flight finish on the previous geometry (the rule of a re-upload, whose cudaFree waits for the device)
    {
        const cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { give_back(); CU(e); }
    }
    BuildReport rep{};
    rc = build_scene_arrays(stg, stg.st, t, p.materials, n, out, s.n_sm, &rep);
    if (rc != CT_OK) {
        // nothing was written when the scratch could not be taken; past that point only a CUDA failure gets here
        give_back();
        return rc;
    }
    lap("scene arrays built on the device");
    void *const old_hot = s.hot_base;
    const size_t old_hot_bytes = s.hot_bytes;
    if (new_hot) { dev_release(s, s.hot_base); s.hot_cap = hl.bytes; }
    if (new_pairs) { dev_release(s, const_cast<DevPair64 *>(p.pairs64)); s.pairs_cap = pairs; }
    if (new_parent) { dev_release(s, s.pair_parent_mem); s.pair_parent_mem = out.pair_parent; s.pair_parent_cap = pairs; }
    if (new_parking) { s.ovf_all = ovf; s.ovf_huge_all = ovf_huge; p.ovf_cap = ovf_cap; p.ovf = ovf; p.ovf_huge = ovf_huge; }
    s.can_overflow = can_overflow;
    s.leaf_dfs_order = true;                                         // BuildBVH's leaves come in DFS order (bvh.cpp:70-97)
    set_tree(s, t, out, rep);
    lap("previous allocations freed");
    if (s.hot_base != old_hot || s.hot_bytes != old_hot_bytes) {
        // the window over the hot records, sized as an upload sizes it, on every stream the frames run on
        release_l2(s);
        TRY(apply_l2_policy(s, device, s.own_stream));
        if (s.stream != s.own_stream) TRY(apply_l2_policy(s, device, s.stream));
        for (cudaStream_t a : s.aux) TRY(apply_l2_policy(s, device, a));
        lap("L2 window re-applied");
    }
    if (timing) fprintf(stderr, "ct_gpu_update_triangles: %u nodes, depth %d, L2 window %zu bytes; total %.2f ms\n", t.n_nodes, t.depth, s.l2_window, now_ms() - t_begin);
    return CT_OK;
}

int ct_gpu_debug_scene_array(int device, const char *name, void *dst, size_t capacity, size_t *bytes) {
    if (!name || !bytes) return fail(CT_ERR_INVALID, "name and bytes must not be NULL");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    const Params &p = s.p;
    ct_scene_summary sum{};
    const void *src = nullptr;
    size_t n = 0;
    const std::string nm(name);
    if (nm == "wide") { src = p.wide; n = (size_t)p.n_wide * sizeof(DevWide); }
    else if (nm == "pairs32") { src = p.pairs32; n = (size_t)p.n_pairs * sizeof(DevPair32); }
    else if (nm == "pairs64") { src = p.pairs64; n = (size_t)p.n_pairs * sizeof(DevPair64); }
    else if (nm == "tris32") { src = p.tris32; n = (size_t)p.n_tri * sizeof(DevTri32); }
    else if (nm == "tris") { src = p.tris; n = (size_t)p.n_tri * sizeof(DevTri); }
    else if (nm == "materials") { src = p.materials; n = (size_t)p.n_tri * sizeof(ct_material); }
    else if (nm == "pair_parent") { src = p.pair_parent; n = p.pair_parent ? (size_t)p.n_pairs * sizeof(uint32_t) : 0; }
    else if (nm == "tri_parent") { src = p.tri_parent; n = (size_t)p.n_tri * sizeof(uint32_t); }
    else if (nm == "summary") {
        sum.n_pairs = p.n_pairs; sum.n_wide = p.n_wide; sum.root_ref = p.root_ref; sum.root_cnt = p.root_cnt; sum.pos_of_tri0 = p.pos_of_tri0;
        sum.nested = p.nested; sum.leaf_dfs_order = s.leaf_dfs_order ? 1u : 0u; sum.can_overflow = s.can_overflow ? 1u : 0u;
        for (int a = 0; a < 3; a++) sum.bound[a] = p.bound[a];
        sum.depth = s.depth;
        n = sizeof sum;
    } else {
        return fail(CT_ERR_INVALID, "unknown scene array \"%s\"", name);
    }
    *bytes = n;
    if (!dst || n == 0) return CT_OK;
    if (capacity < n) return fail(CT_ERR_INVALID, "%s needs %zu bytes, capacity is %zu", name, n, capacity);
    if (nm == "summary") { memcpy(dst, &sum, n); return CT_OK; }
    CU(cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return CT_OK;
}

int ct_gpu_set_camera(int device, const double position[3], const double rotation[9]) {
    if (!position || !rotation) return fail(CT_ERR_INVALID, "NULL camera");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    memcpy(s.p.cam, position, sizeof s.p.cam);
    memcpy(s.p.rot, rotation, sizeof s.p.rot);
    return CT_OK;
}

int ct_gpu_set_stream(int device, void *cuda_stream) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    CU(cudaStreamSynchronize(s.stream));
    if (s.stream != s.own_stream && s.l2_set_aside) {        // take the access-policy window off the caller's previous stream
        cudaStreamAttrValue attr{};
        attr.accessPolicyWindow.num_bytes = 0;
        if (cudaStreamSetAttribute(s.stream, cudaStreamAttributeAccessPolicyWindow, &attr) != cudaSuccess) cudaGetLastError();
    }
    s.stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : s.own_stream;
    TRY(apply_l2_policy(s, device, s.stream));
    return CT_OK;
}

static int render_impl(int device, int y_start, int y_end, ct_ray_counters *counters, bool shared) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    int half = s.p.H / 2;
    // rows outside [-half+?, half] can never be stored (draw2d.h:11): clip so no ray is wasted on them
    int y0 = std::max(y_start, half - (s.p.H - 1)), y1 = std::min(y_end, half + 1);
    if (s.p.subsample) {
        // the partition's own bounds define which rows are traced and averaged (raythread.cpp:457,513,527): no clipping
        if (shared) return fail(CT_ERR_INVALID, "CT_FLAG_SUBSAMPLING needs the whole partition on one device (neighbouring rows are averaged)");
        y0 = y_start; y1 = y_end;
        if (y0 < -(1 << 20) || y1 > (1 << 20)) return fail(CT_ERR_INVALID, "tile [%d,%d) out of range", y_start, y_end);
    }
    if (y1 <= y0) { if (counters) memset(counters, 0, sizeof *counters); return CT_OK; }
    Params p = s.p;
    p.y_lo = y0; p.n_rows = y1 - y0;
    p.n_y = s.p.subsample ? (p.n_rows + 1) / 2 + ((p.n_rows & 1) == 0 ? 1 : 0) : p.n_rows;
    p.n_slots = (uint32_t)p.blocks_x * (uint32_t)((p.n_y + 3) / 4) * 32u * (s.p.supersample ? 16u : 1u);
    if (p.n_slots > p.cap) return fail(CT_ERR_INVALID, "tile [%d,%d) larger than the frame", y_start, y_end);
    const bool count = (s.flags & CT_FLAG_COUNT_TESTS) != 0;
    const int depth_max = s.any_reflective ? p.max_depth : 0;
    // one device: its own cursor (zeroed with the rest of DevSched below) and framebuffer; shared frame: the root's
    // shared frames alternate between two cursors: while frame f steals from cursor f & 1, the root zeroes the other one on
    // its stream for frame f + 1 -- nobody touches that one before the frame-end rendezvous, so no reset call and no
    // host synchronisation stands between two frames
    const bool same_frame = shared && g_hold_frame && s.shared_frames > 0;      // (tests: one device plays several participants of ONE frame)
    const unsigned long long frame_no = same_frame ? s.shared_frames - 1ull : s.shared_frames;
    p.steal = shared ? s.share_cursor + kCursorStride * (frame_no & 1ull) : &p.sched->steal_local;
    const uint32_t shared_shift = g_shared_chunk_shift ? (uint32_t)g_shared_chunk_shift : kChunkSharedShift;
    p.chunk_shift = shared ? shared_shift : kChunkLocalShift;
    p.steal_stride = g_emulate_ranks > 1 ? (uint32_t)g_emulate_ranks : 1u;
    if (p.steal_stride > 1) p.chunk_shift = shared_shift;
    const bool dealt = shared && p.steal_stride == 1 && s.part_count > 1;
    p.part_index = dealt ? (uint32_t)s.part_index : 0u;
    p.part_count = dealt ? (uint32_t)s.part_count : 0u;
    p.static_eighths = (uint32_t)g_static_eighths;
    p.run_shift = (shared || p.steal_stride > 1) ? (uint32_t)g_run_shift : 0u;
    if (shared && !s.remote_cursor_ok) {
        // no native atomics to the root's cursor: stealing from it would hand chunks out twice or not at all
        if (!dealt) return fail(CT_ERR_CUDA, "device %d has no native atomics to the shared frame's cursor: declare the participants (ct_gpu_share_partition), then every chunk is dealt", device);
        p.static_eighths = 8u;
    }
    p.fb_out = shared ? s.share_fb : p.fb;
    Params pk = p; pk.max_depth = depth_max;   // with no reflective material the recursion never goes past depth 0 (:369)
    pk.parent_q_all = s.parent_q_all; pk.hitb_t_all = s.hitb_t_all; pk.occ_all = s.occ_all;
    pk.reuse_shadow = (g_shadow_reuse && s.parent_q_all) ? 1u : 0u;
    cudaStream_t st = s.stream;
    if (shared && !same_frame) {
        if (s.share_cursor == s.cursor_own) CU(cudaMemsetAsync(s.cursor_own + kCursorStride * ((s.shared_frames + 1ull) & 1ull), 0, sizeof(unsigned long long), st));
        s.shared_frames++;
    }
    CU(cudaMemsetAsync(p.sched, 0, sizeof(DevSched), st));
    CU(cudaEventRecord(s.ev0, st));
    const bool stages = (s.flags & CT_FLAG_STAGE_TIMING) != 0;
    s.n_stages = 0;
    if (stages) CU(cudaEventRecord(s.stage_ev[0], st));
    auto mark = [&](const char *name, int depth) -> int {          // called after each launch on st
        s.launches++;
        if (!stages || s.n_stages >= kMaxLaunches) return CT_OK;
        s.stage_name[s.n_stages] = name; s.stage_depth[s.n_stages] = depth;
        s.n_stages++;
        CU(cudaEventRecord(s.stage_ev[s.n_stages], st));
        return CT_OK;
    };
    const PathArrays arrays{s.hitb_t_all, s.hitb_pos_all, s.rays_all, s.path_slot_all, s.occ_all, s.parent_q_all, s.far_all,
                            s.ovf_all, s.ovf_huge_all};
    TRY(enqueue_stages<false>(s, pk, arrays, count, stages, st, mark, s.launches));
    CU(cudaEventRecord(s.ev1, st));
    CU(cudaEventRecord(s.tile_done[s.tiles_submitted % 8], st));
    s.tiles_submitted++;
    CU(cudaGetLastError());
    s.timed = true;
    {   // framebuffer rows this tile writes: row = H/2 - y
        int lo = half - (y1 - 1), hi = half - y0 + 1 + (s.p.subsample ? 1 : 0);   // subsampling also stores row y0 - 1
        lo = std::max(lo, 0); hi = std::min(hi, s.p.H);
        extend_rows(s, lo, hi);
    }
    if (counters) {
        ct_ray_counters now;
        TRY(read_totals(s, &now));
        counters->rays_primary = now.rays_primary - s.snapshot.rays_primary;
        counters->rays_shadow = now.rays_shadow - s.snapshot.rays_shadow;
        counters->rays_reflection = now.rays_reflection - s.snapshot.rays_reflection;
        counters->box_tests = now.box_tests - s.snapshot.box_tests;
        counters->tri_tests = now.tri_tests - s.snapshot.tri_tests;
        s.snapshot = now;
    }
    return CT_OK;
}

int ct_gpu_render_tile(int device, int y_start, int y_end, ct_ray_counters *counters) {
    return render_impl(device, y_start, y_end, counters, false);
}

int ct_gpu_render_shared(int device, int y_start, int y_end, ct_ray_counters *counters) {
    return render_impl(device, y_start, y_end, counters, true);
}

int ct_gpu_share_export(int device, ct_gpu_share *out) {
    if (!out || out->struct_size != sizeof(ct_gpu_share)) return fail(CT_ERR_INVALID, "ct_gpu_share missing or struct_size != %zu", sizeof(ct_gpu_share));
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ct_gpu_share reserves 64 bytes per IPC handle");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, s.p.fb));
    memcpy(out->fb_ipc, &h, sizeof h);
    CU(cudaIpcGetMemHandle(&h, s.cursor_own));
    memcpy(out->cursor_ipc, &h, sizeof h);
    out->device = device;
    out->pid = (int64_t)getpid();
    out->fb_ptr = (uint64_t)(uintptr_t)s.p.fb;
    out->cursor_ptr = (uint64_t)(uintptr_t)s.cursor_own;
    out->width = s.p.W; out->height = s.p.H;
    out->frames = s.shared_frames;
    return CT_OK;
}

int ct_gpu_share_attach(int device, const ct_gpu_share *root) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    for (void *&q : s.ipc_opened) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    s.remote_cursor_ok = true;
    if (root) s.shared_frames = root->frames;                // which of the two cursors the next shared frame uses
    if (!root) {                                             // detach: back to this device's own cursor and framebuffer
        s.share_cursor = s.cursor_own; s.share_fb = s.p.fb;
        return CT_OK;
    }
    if (root->struct_size != sizeof(ct_gpu_share)) return fail(CT_ERR_INVALID, "ct_gpu_share struct_size != %zu", sizeof(ct_gpu_share));
    if (root->width != s.p.W || root->height != s.p.H) return fail(CT_ERR_INVALID, "shared frame is %dx%d, this device renders %dx%d", root->width, root->height, s.p.W, s.p.H);
    if (root->device != device) {
        // next_chunk steals with atomicAdd on the root's cursor: across devices that is only atomic where the link has
        // native atomics (NVLink; not PCIe peer access).  Without them this device takes dealt chunks only (render_impl).
        int native = 0;
        if (cudaDeviceGetP2PAttribute(&native, cudaDevP2PAttrNativeAtomicSupported, device, root->device) != cudaSuccess) { cudaGetLastError(); native = 0; }
        s.remote_cursor_ok = native != 0;
    }
    if (root->pid == (int64_t)getpid()) {                    // same process: raw pointers (+ peer access between the two devices)
        if (root->device != device) {
            int can = 0;
            CU(cudaDeviceCanAccessPeer(&can, device, root->device));
            if (!can) return fail(CT_ERR_CUDA, "device %d cannot access device %d's memory", device, root->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(CT_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
        s.share_fb = (uint32_t *)(uintptr_t)root->fb_ptr;
        s.share_cursor = (unsigned long long *)(uintptr_t)root->cursor_ptr;
        return CT_OK;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, root->fb_ipc, sizeof h);
    CU(cudaIpcOpenMemHandle(&s.ipc_opened[0], h, cudaIpcMemLazyEnablePeerAccess));
    memcpy(&h, root->cursor_ipc, sizeof h);
    CU(cudaIpcOpenMemHandle(&s.ipc_opened[1], h, cudaIpcMemLazyEnablePeerAccess));
    s.share_fb = (uint32_t *)s.ipc_opened[0];
    s.share_cursor = (unsigned long long *)s.ipc_opened[1];
    return CT_OK;
}

int ct_gpu_share_partition(int device, int index, int count) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (count < 0 || count > 64 || (count > 0 && (index < 0 || index >= count))) return fail(CT_ERR_INVALID, "bad partition %d of %d", index, count);
    s.part_index = count > 1 ? index : 0;
    s.part_count = count > 1 ? count : 0;
    return CT_OK;
}

int ct_gpu_share_reset(int device) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    CU(cudaMemsetAsync(s.cursor_own, 0, 2 * kCursorStride * sizeof(unsigned long long), s.stream));
    CU(cudaStreamSynchronize(s.stream));
    return CT_OK;
}

int ct_gpu_set_option(const char *name, long long value) {
    if (!name) return fail(CT_ERR_INVALID, "NULL option name");
    if (!strcmp(name, "traversal_budget")) {
        if (value < 0) return fail(CT_ERR_INVALID, "traversal_budget must be >= 0 (0 = default)");
        g_budget_option = value;
        return CT_OK;
    }
    if (!strcmp(name, "emulate_ranks")) {
        if (value < 0 || value > 64) return fail(CT_ERR_INVALID, "emulate_ranks must be 0..64");
        g_emulate_ranks = value;
        return CT_OK;
    }
    if (!strcmp(name, "shared_static_eighths")) {
        if (value < 0 || value > 8) return fail(CT_ERR_INVALID, "shared_static_eighths must be 0..8");
        g_static_eighths = value;
        return CT_OK;
    }
    if (!strcmp(name, "shared_chunk_shift")) {
        if (value != 0 && (value < kChunkLocalShift || value > kChunkMaxShift)) return fail(CT_ERR_INVALID, "shared_chunk_shift must be 0 (default), 5 or 6");
        g_shared_chunk_shift = value;
        return CT_OK;
    }
    if (!strcmp(name, "shared_run_shift")) {
        if (value < 0 || value > 10) return fail(CT_ERR_INVALID, "shared_run_shift must be 0..10");
        g_run_shift = value;
        return CT_OK;
    }
    if (!strcmp(name, "shadow_reuse")) {
        if (value != 0 && value != 1) return fail(CT_ERR_INVALID, "shadow_reuse must be 0 or 1");
        g_shadow_reuse = value;
        return CT_OK;
    }
    if (!strcmp(name, "shared_hold_frame")) {
        if (value != 0 && value != 1) return fail(CT_ERR_INVALID, "shared_hold_frame must be 0 or 1");
        g_hold_frame = value;
        return CT_OK;
    }
    if (!strcmp(name, "l2_persist")) {
        if (value != 0 && value != 1) return fail(CT_ERR_INVALID, "l2_persist must be 0 or 1");
        g_l2_persist = value;
        return CT_OK;
    }
    if (!strcmp(name, "any_leaves")) {
        if (value != 0 && (value < 5 || value > 64)) return fail(CT_ERR_INVALID, "any_leaves must be 0 (default) or 5..64");
        g_any_leaves = value;
        return CT_OK;
    }
    if (!strcmp(name, "primary_split")) {
        if (value != 0 && value != 1) return fail(CT_ERR_INVALID, "primary_split must be 0 or 1");
        g_primary_split = value;
        return CT_OK;
    }
    if (!strcmp(name, "primary_budget")) {
        g_primary_budget_option = value;
        return CT_OK;
    }
    if (!strcmp(name, "overflow_warp_budget")) {
        if (value < 0) return fail(CT_ERR_INVALID, "overflow_warp_budget must be >= 0 (0 = default)");
        g_warp_budget_option = value;
        return CT_OK;
    }
    return fail(CT_ERR_INVALID, "unknown option '%s'", name);
}

int ct_gpu_overflow_stats(int device, uint64_t *parked, uint64_t *finished_in_place) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    ct_ray_counters tmp;
    TRY(read_totals(s, &tmp));
    if (parked) *parked = s.rays_overflow;
    if (finished_in_place) *finished_in_place = s.rays_in_place;
    return CT_OK;
}

int ct_gpu_reuse_stats(int device, uint64_t *shadow_rays_reused) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    ct_ray_counters tmp;
    TRY(read_totals(s, &tmp));
    if (shadow_rays_reused) *shadow_rays_reused = s.rays_shadow_reused;
    return CT_OK;
}

int ct_gpu_filter_stats(int device, uint64_t *box_exact, uint64_t *tri_exact) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    ct_ray_counters tmp;
    TRY(read_totals(s, &tmp));
    if (box_exact) *box_exact = s.box_exact;
    if (tri_exact) *tri_exact = s.tri_exact;
    return CT_OK;
}

int ct_gpu_sync(int device) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    CU(cudaStreamSynchronize(s.stream));
    return CT_OK;
}

int ct_gpu_kernel_launches(int device, uint64_t *out, int reset) {
    if (!out) return fail(CT_ERR_INVALID, "NULL out");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    *out = s.launches;
    if (reset) s.launches = 0;
    return CT_OK;
}

int ct_gpu_last_tile_stages(int device, int max, float *ms, const char **names, int *depth) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (!(s.flags & CT_FLAG_STAGE_TIMING)) return fail(CT_ERR_INVALID, "scene was uploaded without CT_FLAG_STAGE_TIMING");
    CU(cudaStreamSynchronize(s.stream));
    for (int i = 0; i < s.n_stages && i < max; i++) {
        if (ms) CU(cudaEventElapsedTime(&ms[i], s.stage_ev[i], s.stage_ev[i + 1]));
        if (names) names[i] = s.stage_name[i];
        if (depth) depth[i] = s.stage_depth[i];
    }
    return s.n_stages;
}

int ct_gpu_throttle(int device, int max_in_flight) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (max_in_flight <= 0) { CU(cudaStreamSynchronize(s.stream)); return CT_OK; }
    unsigned long long keep = (unsigned long long)std::min(max_in_flight, 7);
    if (s.tiles_submitted > keep) CU(cudaEventSynchronize(s.tile_done[(s.tiles_submitted - keep - 1) % 8]));
    return CT_OK;
}

int ct_gpu_last_tile_ms(int device, float *ms) {
    if (!ms) return fail(CT_ERR_INVALID, "NULL ms");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded || !s.timed) return fail(CT_ERR_NO_SCENE, "no tile rendered on device %d", device);
    CU(cudaEventSynchronize(s.ev1));
    CU(cudaEventElapsedTime(ms, s.ev0, s.ev1));
    return CT_OK;
}

int ct_gpu_get_counters(int device, ct_ray_counters *out, int reset) {
    if (!out) return fail(CT_ERR_INVALID, "NULL out");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    TRY(read_totals(s, out));
    if (reset) {
        CU(cudaMemset(s.p.tot, 0, sizeof(DevTotals)));
        s.snapshot = ct_ray_counters{};
    }
    return CT_OK;
}

int ct_gpu_readback(int device, uint32_t *dst, int dst_stride_pixels, int row_start, int row_end) {
    if (!dst) return fail(CT_ERR_INVALID, "NULL dst");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    const Params &p = s.p;
    // Only rows some tile has rendered are copied: e.g. row 0 (y = H/2) is never reached by the reference's
    // loops (y < yEnd <= H/2, SURVEY 0.6) and so stays untouched in dst here as well.
    int row_lo, row_hi;
    { std::lock_guard<std::mutex> lock(g_rows_mutex); row_lo = s.row_lo; row_hi = s.row_hi; }
    int r0 = std::max(row_start, row_lo), r1 = std::min(row_end, row_hi);
    int cols = s.col_hi - s.col_lo;
    if (dst_stride_pixels < p.W) return fail(CT_ERR_INVALID, "dst stride %d < width %d", dst_stride_pixels, p.W);
    CU(cudaStreamSynchronize(s.stream));
    if (r1 <= r0 || cols <= 0) return CT_OK;
    CU(cudaMemcpy2D(dst + (size_t)r0 * dst_stride_pixels + s.col_lo, (size_t)dst_stride_pixels * 4,
                    p.fb + (size_t)r0 * p.W + s.col_lo, (size_t)p.W * 4, (size_t)cols * 4, (size_t)(r1 - r0),
                    cudaMemcpyDeviceToHost));
    return CT_OK;
}

int ct_gpu_readback_async(int device, uint32_t *dst, int dst_stride_pixels, int row_start, int row_end) {
    if (!dst) return fail(CT_ERR_INVALID, "NULL dst");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    const Params &p = s.p;
    if (dst_stride_pixels < p.W) return fail(CT_ERR_INVALID, "dst stride %d < width %d", dst_stride_pixels, p.W);
    if (!s.copy_stream) {
        TRY(dev_alloc(s, &s.fb_snapshot, (size_t)p.W * p.H));
        CU(cudaStreamCreateWithFlags(&s.copy_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&s.ev_snap, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_copied, cudaEventDisableTiming));
    }
    int row_lo, row_hi;
    { std::lock_guard<std::mutex> lock(g_rows_mutex); row_lo = s.row_lo; row_hi = s.row_hi; }
    const int r0 = std::max(row_start, row_lo), r1 = std::min(row_end, row_hi), cols = s.col_hi - s.col_lo;
    // in stream order behind the tiles submitted so far: snapshot the rows on the device (microseconds), so that the next
    // frame may overwrite the framebuffer while the copy stream moves the snapshot to the host (PCIe, ~0.4 ms for a 4K frame)
    if (s.copy_pending) CU(cudaStreamWaitEvent(s.stream, s.ev_copied, 0));       // the previous snapshot has left the device
    if (r1 > r0 && cols > 0)
        CU(cudaMemcpy2DAsync(s.fb_snapshot + (size_t)r0 * p.W + s.col_lo, (size_t)p.W * 4, p.fb + (size_t)r0 * p.W + s.col_lo, (size_t)p.W * 4,
                             (size_t)cols * 4, (size_t)(r1 - r0), cudaMemcpyDeviceToDevice, s.stream));
    CU(cudaEventRecord(s.ev_snap, s.stream));
    CU(cudaStreamWaitEvent(s.copy_stream, s.ev_snap, 0));
    if (r1 > r0 && cols > 0)
        CU(cudaMemcpy2DAsync(dst + (size_t)r0 * dst_stride_pixels + s.col_lo, (size_t)dst_stride_pixels * 4,
                             s.fb_snapshot + (size_t)r0 * p.W + s.col_lo, (size_t)p.W * 4, (size_t)cols * 4, (size_t)(r1 - r0),
                             cudaMemcpyDeviceToHost, s.copy_stream));
    CU(cudaEventRecord(s.ev_copied, s.copy_stream));
    s.copy_pending = true;
    return CT_OK;
}

int ct_gpu_readback_wait(int device) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (s.copy_pending) CU(cudaEventSynchronize(s.ev_copied));
    s.copy_pending = false;
    return CT_OK;
}

int ct_gpu_readback_hits(int device, uint32_t *found, uint32_t *index, float *t, int stride_pixels, int row_start, int row_end) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    const Params &p = s.p;
    if (!p.dbg_found) return fail(CT_ERR_INVALID, "scene was uploaded without CT_FLAG_KEEP_HITS");
    if (stride_pixels < p.W) return fail(CT_ERR_INVALID, "stride %d < width %d", stride_pixels, p.W);
    int r0 = std::max(row_start, 0), r1 = std::min(row_end, p.H);
    CU(cudaStreamSynchronize(s.stream));
    if (r1 <= r0) return CT_OK;
    size_t rows = (size_t)(r1 - r0);
    if (found) CU(cudaMemcpy2D(found + (size_t)r0 * stride_pixels, (size_t)stride_pixels * 4, p.dbg_found + (size_t)r0 * p.W, (size_t)p.W * 4, (size_t)p.W * 4, rows, cudaMemcpyDeviceToHost));
    if (index) CU(cudaMemcpy2D(index + (size_t)r0 * stride_pixels, (size_t)stride_pixels * 4, p.dbg_index + (size_t)r0 * p.W, (size_t)p.W * 4, (size_t)p.W * 4, rows, cudaMemcpyDeviceToHost));
    if (t) CU(cudaMemcpy2D(t + (size_t)r0 * stride_pixels, (size_t)stride_pixels * 4, p.dbg_t + (size_t)r0 * p.W, (size_t)p.W * 4, (size_t)p.W * 4, rows, cudaMemcpyDeviceToHost));
    return CT_OK;
}

int ct_gpu_framebuffer(int device, void **device_ptr, int *width, int *height) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (device_ptr) *device_ptr = s.p.fb;
    if (width) *width = s.p.W;
    if (height) *height = s.p.H;
    return CT_OK;
}

int ct_gpu_gather_rows(int src_device, int dst_device, int row_start, int row_end) {
    TRY(check_device(dst_device));
    TRY(check_device(src_device));
    DeviceState &a = g_dev[src_device], &b = g_dev[dst_device];
    if (!a.loaded || !b.loaded) return fail(CT_ERR_NO_SCENE, "both devices need an uploaded scene");
    if (a.p.W != b.p.W || a.p.H != b.p.H) return fail(CT_ERR_INVALID, "frame sizes differ between devices");
    int r0 = std::max(row_start, 0), r1 = std::min(row_end, a.p.H);
    if (r1 <= r0 || src_device == dst_device) return CT_OK;
    size_t off = (size_t)r0 * a.p.W, bytes = (size_t)(r1 - r0) * a.p.W * 4;
    CU(cudaMemcpyPeerAsync(b.p.fb + off, dst_device, a.p.fb + off, src_device, bytes, a.stream));
    extend_rows(b, r0, r1);                 // the destination's readback must cover rows it did not render itself
    return CT_OK;
}

int ct_gpu_mark_rows(int device, int row_start, int row_end) {
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    int r0 = std::max(row_start, 0), r1 = std::min(row_end, s.p.H);
    if (r1 > r0) extend_rows(s, r0, r1);
    return CT_OK;
}

int ct_gpu_debug_closest(int device, uint32_t n, const double *origins, const double *directions, const float *t0,
                         uint32_t *found, uint32_t *index, float *tclosest) {
    if (!origins || !directions || !t0) return fail(CT_ERR_INVALID, "NULL ray arrays");
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (n == 0) return CT_OK;
    double *d_o = nullptr, *d_d = nullptr; float *d_t0 = nullptr, *d_tc = nullptr; uint32_t *d_f = nullptr, *d_i = nullptr;
    int rc = CT_OK;
    auto cleanup = [&]() { cudaFree(d_o); cudaFree(d_d); cudaFree(d_t0); cudaFree(d_tc); cudaFree(d_f); cudaFree(d_i); };
#define CUX(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(CT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); cleanup(); return rc; } } while (0)
    CUX(cudaMalloc(&d_o, 24ull * n)); CUX(cudaMalloc(&d_d, 24ull * n)); CUX(cudaMalloc(&d_t0, 4ull * n));
    CUX(cudaMalloc(&d_tc, 4ull * n)); CUX(cudaMalloc(&d_f, 4ull * n)); CUX(cudaMalloc(&d_i, 4ull * n));
    CUX(cudaMemcpy(d_o, origins, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_d, directions, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_t0, t0, 4ull * n, cudaMemcpyHostToDevice));
    CUX(cudaStreamSynchronize(s.stream));
    k_debug_closest<<<(n + kBlockThreads - 1) / kBlockThreads, kBlockThreads, 0, s.stream>>>(s.p, n, d_o, d_d, d_t0, d_f, d_i, d_tc);
    CUX(cudaGetLastError());
    CUX(cudaStreamSynchronize(s.stream));
    if (found) CUX(cudaMemcpy(found, d_f, 4ull * n, cudaMemcpyDeviceToHost));
    if (index) CUX(cudaMemcpy(index, d_i, 4ull * n, cudaMemcpyDeviceToHost));
    if (tclosest) CUX(cudaMemcpy(tclosest, d_tc, 4ull * n, cudaMemcpyDeviceToHost));
    cleanup();
    return CT_OK;
}

int ct_gpu_debug_early(int device, int mode, uint32_t n, const double *origins, const double *directions,
                       uint32_t *found, uint32_t *index, uint32_t *path) {
    if (!origins || !directions) return fail(CT_ERR_INVALID, "NULL ray arrays");
    if (mode != 0 && mode != 1) return fail(CT_ERR_INVALID, "mode must be 0 (shadow ray) or 1 (reflection ray)");
    return debug_query(device, mode == 0 ? CT_RAY_SHADOW : CT_RAY_REFLECTION, n, origins, directions, 0u, found, index, nullptr, path);
}

int ct_gpu_debug_primary(int device, uint32_t n, const double *origins, const double *directions, uint32_t park_cap,
                         uint32_t *found, uint32_t *index, float *tclosest, uint32_t *path) {
    if (!origins || !directions) return fail(CT_ERR_INVALID, "NULL ray arrays");
    return debug_query(device, CT_RAY_PRIMARY, n, origins, directions, park_cap, found, index, tclosest, path);
}

int ct_gpu_trace_rays(int device, const ct_ray_query *q) {
    if (!q || q->struct_size != sizeof(ct_ray_query)) return fail(CT_ERR_INVALID, "ct_ray_query missing or struct_size != %zu", sizeof(ct_ray_query));
    if (q->kind != CT_RAY_PRIMARY && q->kind != CT_RAY_SHADOW && q->kind != CT_RAY_REFLECTION) return fail(CT_ERR_INVALID, "unknown ray kind %d", q->kind);
    if (q->n >= (1u << 31)) return fail(CT_ERR_LIMIT, "%u rays: a query takes fewer than 2^31", q->n);
    if (q->n > 0 && (!q->origins || !q->directions)) return fail(CT_ERR_INVALID, "NULL origins or directions with n = %u", q->n);
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (q->n == 0) return CT_OK;
    const struct { const void *p; size_t align; const char *name; } arrays[] = {
        {q->origins, 8, "origins"}, {q->directions, 8, "directions"}, {q->found, 4, "found"}, {q->index, 4, "index"}, {q->tclosest, 4, "tclosest"}};
    for (const auto &a : arrays)
        if (a.p) TRY(check_device_array(device, a.p, a.align, a.name));
    const cudaStream_t st = q->stream ? static_cast<cudaStream_t>(q->stream) : s.stream;
    const bool shadow = q->kind == CT_RAY_SHADOW;
    return trace_impl(s, q->kind, q->n, q->origins, q->directions, q->found, shadow ? nullptr : q->index, shadow ? nullptr : q->tclosest,
                      nullptr, 0u, st);
}

int ct_gpu_shade_rays(int device, const ct_shade_query *q) {
    if (!q || q->struct_size != sizeof(ct_shade_query)) return fail(CT_ERR_INVALID, "ct_shade_query missing or struct_size != %zu", sizeof(ct_shade_query));
    if (q->n >= (1u << 31)) return fail(CT_ERR_LIMIT, "%u rays: a query takes fewer than 2^31", q->n);
    if (q->max_depth > 15) return fail(CT_ERR_LIMIT, "max_depth %d outside 0..15 (< 0: the scene's)", q->max_depth);
    if (q->n > 0 && (!q->origins || !q->directions || !q->color)) return fail(CT_ERR_INVALID, "NULL origins, directions or color with n = %u", q->n);
    TRY(check_device(device));
    DEVICE_GUARD(device);
    DeviceState &s = g_dev[device];
    if (!s.loaded) return fail(CT_ERR_NO_SCENE, "no scene uploaded on device %d", device);
    if (q->n == 0) return CT_OK;
    TRY(check_device_array(device, q->origins, 8, "origins"));
    TRY(check_device_array(device, q->directions, 8, "directions"));
    TRY(check_device_array(device, q->color, 4, "color"));
    const cudaStream_t st = q->stream ? static_cast<cudaStream_t>(q->stream) : s.stream;
    return shade_impl(s, q->n, q->max_depth < 0 ? s.p.max_depth : q->max_depth, q->origins, q->directions, q->color, st);
}

static int debug_primitives_impl(int device, uint32_t n, const double *origins, const double *directions, float *ray_t,
                                 const double *tri, const double *bmin, const double *bmax, uint32_t *tri_hit, uint32_t *box_hit,
                                 uint32_t *filter_out, double bound_scale, bool keep_ray_t = false) {
    TRY(check_device(device));
    if (n == 0) return CT_OK;
    double *d_o = nullptr, *d_d = nullptr, *d_tri = nullptr, *d_mn = nullptr, *d_mx = nullptr; float *d_t = nullptr;
    uint32_t *d_th = nullptr, *d_bh = nullptr, *d_f = nullptr;
    int rc = CT_OK;
    auto cleanup = [&]() { cudaFree(d_o); cudaFree(d_d); cudaFree(d_tri); cudaFree(d_mn); cudaFree(d_mx); cudaFree(d_t); cudaFree(d_th); cudaFree(d_bh); cudaFree(d_f); };
    CUX(cudaMalloc(&d_o, 24ull * n)); CUX(cudaMalloc(&d_d, 24ull * n)); CUX(cudaMalloc(&d_tri, 72ull * n));
    CUX(cudaMalloc(&d_mn, 24ull * n)); CUX(cudaMalloc(&d_mx, 24ull * n)); CUX(cudaMalloc(&d_t, 4ull * n));
    CUX(cudaMalloc(&d_th, 4ull * n)); CUX(cudaMalloc(&d_bh, 4ull * n));
    if (filter_out) CUX(cudaMalloc(&d_f, 4ull * n));
    CUX(cudaMemcpy(d_o, origins, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_d, directions, 24ull * n, cudaMemcpyHostToDevice));
    if (tri) CUX(cudaMemcpy(d_tri, tri, 72ull * n, cudaMemcpyHostToDevice));
    else CUX(cudaMemset(d_tri, 0, 72ull * n));
    CUX(cudaMemcpy(d_mn, bmin, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_mx, bmax, 24ull * n, cudaMemcpyHostToDevice));
    CUX(cudaMemcpy(d_t, ray_t, 4ull * n, cudaMemcpyHostToDevice));
    k_debug_primitives<<<(n + 127) / 128, 128>>>(n, d_o, d_d, d_t, d_tri, d_mn, d_mx, d_th, d_bh, d_f, bound_scale, filter_out != nullptr && tri != nullptr);
    CUX(cudaGetLastError());
    CUX(cudaDeviceSynchronize());
    if (tri && !keep_ray_t) CUX(cudaMemcpy(ray_t, d_t, 4ull * n, cudaMemcpyDeviceToHost));
    if (tri_hit) CUX(cudaMemcpy(tri_hit, d_th, 4ull * n, cudaMemcpyDeviceToHost));
    if (box_hit) CUX(cudaMemcpy(box_hit, d_bh, 4ull * n, cudaMemcpyDeviceToHost));
    if (filter_out) CUX(cudaMemcpy(filter_out, d_f, 4ull * n, cudaMemcpyDeviceToHost));
    cleanup();
#undef CUX
    return CT_OK;
}

int ct_gpu_debug_primitives(int device, uint32_t n, const double *origins, const double *directions, float *ray_t,
                            const double *tri, const double *bmin, const double *bmax, uint32_t *tri_hit, uint32_t *box_hit) {
    if (!origins || !directions || !ray_t || !tri || !bmin || !bmax || !tri_hit || !box_hit) return fail(CT_ERR_INVALID, "NULL array");
    return debug_primitives_impl(device, n, origins, directions, ray_t, tri, bmin, bmax, tri_hit, box_hit, nullptr, 1.0);
}

int ct_gpu_debug_filter(int device, uint32_t n, const double *origins, const double *directions, const float *ray_t,
                        const double *tri, const double *bmin, const double *bmax, double bound_scale, uint32_t *verdict) {
    if (!origins || !directions || !ray_t || !bmin || !bmax || !verdict) return fail(CT_ERR_INVALID, "NULL array");
    if (!(bound_scale >= 1.0)) return fail(CT_ERR_INVALID, "bound_scale must be >= 1");
    return debug_primitives_impl(device, n, origins, directions, const_cast<float *>(ray_t), tri, bmin, bmax, nullptr, nullptr, verdict, bound_scale, true);
}

int ct_gpu_debug_shading(int device, uint32_t n, const uint32_t *color, const float *intensity, uint32_t *shaded,
                         const uint32_t *lc, const uint32_t *rc, const float *reflection, uint32_t *blended,
                         const float *x, const int32_t *e, double *pow_out, const float *acc, const float *li, float *acc_out) {
    if ((shaded && (!color || !intensity)) || (blended && (!lc || !rc || !reflection)) || ((pow_out || acc_out) && (!x || !e)) ||
        (acc_out && (!acc || !li)))
        return fail(CT_ERR_INVALID, "NULL input for a requested output");
    TRY(check_device(device));
    if (n == 0) return CT_OK;
    std::vector<void *> bufs;
    int rc_ = CT_OK;
    auto cleanup = [&]() { for (void *p : bufs) cudaFree(p); };
#define CUX(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc_ = fail(CT_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); cleanup(); return rc_; } } while (0)
    // a device copy of n elements of `src` (uploaded when given), nullptr when the family is not requested
    auto dev = [&](const void *src, size_t elem, bool want, void **out) -> cudaError_t {
        *out = nullptr;
        if (!want) return cudaSuccess;
        cudaError_t err = cudaMalloc(out, elem * n);
        if (err != cudaSuccess) return err;
        bufs.push_back(*out);
        return src ? cudaMemcpy(*out, src, elem * n, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    const bool want_pow = pow_out || acc_out;
    void *d_color, *d_int, *d_shaded, *d_lc, *d_rc, *d_refl, *d_blended, *d_x, *d_e, *d_pow, *d_acc, *d_li, *d_acc_out;
    CUX(dev(color, 4, shaded, &d_color)); CUX(dev(intensity, 4, shaded, &d_int)); CUX(dev(nullptr, 4, shaded, &d_shaded));
    CUX(dev(lc, 4, blended, &d_lc)); CUX(dev(rc, 4, blended, &d_rc)); CUX(dev(reflection, 4, blended, &d_refl)); CUX(dev(nullptr, 4, blended, &d_blended));
    CUX(dev(x, 4, want_pow, &d_x)); CUX(dev(e, 4, want_pow, &d_e)); CUX(dev(nullptr, 8, pow_out, &d_pow));
    CUX(dev(acc, 4, acc_out, &d_acc)); CUX(dev(li, 4, acc_out, &d_li)); CUX(dev(nullptr, 4, acc_out, &d_acc_out));
    k_debug_shading<<<(n + 255) / 256, 256>>>(n, (const uint32_t *)d_color, (const float *)d_int, (uint32_t *)d_shaded,
                                               (const uint32_t *)d_lc, (const uint32_t *)d_rc, (const float *)d_refl, (uint32_t *)d_blended,
                                               (const float *)d_x, (const int32_t *)d_e, (double *)d_pow, (const float *)d_acc, (const float *)d_li,
                                               (float *)d_acc_out);
    CUX(cudaGetLastError());
    CUX(cudaDeviceSynchronize());
    if (shaded) CUX(cudaMemcpy(shaded, d_shaded, 4ull * n, cudaMemcpyDeviceToHost));
    if (blended) CUX(cudaMemcpy(blended, d_blended, 4ull * n, cudaMemcpyDeviceToHost));
    if (pow_out) CUX(cudaMemcpy(pow_out, d_pow, 8ull * n, cudaMemcpyDeviceToHost));
    if (acc_out) CUX(cudaMemcpy(acc_out, d_acc_out, 4ull * n, cudaMemcpyDeviceToHost));
    cleanup();
#undef CUX
    return CT_OK;
}

int ct_gpu_shutdown(int device) {
    if (device < 0 || device >= kMaxDevices) return fail(CT_ERR_NO_DEVICE, "device %d out of range", device);
    DEVICE_GUARD(device);
    std::lock_guard<std::mutex> lock(g_mutex);
    DeviceState &s = g_dev[device];
    if (s.loaded || !s.allocs.empty()) {
        cudaSetDevice(device);
        cudaDeviceSynchronize();
        free_device(s);
    }
    return CT_OK;
}

}  // extern "C"
