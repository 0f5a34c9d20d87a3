/* include/ct_gpu.h -- C ABI of the B200 renderer that sits behind CobbleTrace's boss/worker
 * entry point (reference raythread.cpp:641 RayThread; SURVEY.md 8b).
 *
 * Everything is plain C: POD structs, pointers and sizes.  Every function returns 0 on
 * success or a negative ct_status; nothing calls exit() (the reference's workers do:
 * raythread.cpp:591,608).  ct_gpu_last_error() gives a message for the calling thread.
 * The library copies at upload and never keeps a host pointer past the call that received
 * it.  There is no CPU fallback: without a CUDA device every compute call fails with
 * CT_ERR_NO_DEVICE.
 *
 * Struct layouts deliberately equal the reference's in-memory layouts on x86-64
 * (sizeof checked in SURVEY 8: bvh_node_t 64, light_t 56, material_t 12), so a binding
 * can pass the reference's own arrays without repacking; see INTEGRATION.md.
 *
 * Threading: one host thread per device at a time.  Work is asynchronous on one CUDA
 * stream per device; ct_gpu_readback(_hits), ct_gpu_get_counters and ct_gpu_sync are the
 * synchronisation points that replace the reference's WS_FINISHED polling
 * (raythread.cpp:657-661).
 */
#ifndef CT_GPU_H
#define CT_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CT_GPU_ABI_VERSION 1

typedef enum ct_status {
    CT_OK = 0,
    CT_ERR_INVALID = -1,      /* bad argument / descriptor */
    CT_ERR_NO_DEVICE = -2,    /* no CUDA device, or device index out of range */
    CT_ERR_CUDA = -3,         /* a CUDA runtime call failed (see ct_gpu_last_error) */
    CT_ERR_NO_SCENE = -4,     /* render/readback before a successful upload */
    CT_ERR_LIMIT = -5,        /* scene exceeds a device-side limit (BVH depth, counts) */
    CT_ERR_OOM = -6           /* device allocation failed */
} ct_status;

/* == bvh_node_t, reference bvh.h:5-11 (two v3_t of double, three uint32, 4 bytes tail padding) */
typedef struct ct_bvh_node {
    double aabb_min[3];
    double aabb_max[3];
    uint32_t left_node;             /* children are left_node and left_node+1 (bvh.cpp:89-97) */
    uint32_t first_triangle_index;  /* into tri_indexes */
    uint32_t triangle_count;        /* 0 = interior (bvh.cpp:99) */
    uint32_t _pad;
} ct_bvh_node;

/* == material_t, reference scenefile.h:25-29 */
typedef struct ct_material {
    uint32_t color;      /* 0x00BBGGRR, color.h:77-80 */
    int32_t specular;    /* -1 disables the specular term (raythread.cpp:316) */
    float reflection;    /* <= 0 stops recursion (raythread.cpp:369) */
} ct_material;

/* == light_t, reference scenefile.h:61-66; type values == lightType_t scenefile.h:13 */
enum { CT_LIGHT_POINT = 0, CT_LIGHT_DIRECTIONAL = 1, CT_LIGHT_AMBIENT = 2 };
typedef struct ct_light {
    int32_t type;
    float intensity;
    double position[3];
    double direction[3];
} ct_light;

enum {
    CT_FLAG_WIDE = 1u,        /* trace x in [-W/2, W/2) instead of the reference's centred HxH square
                                 (raythread.cpp:454-455 "Keep it square"); SURVEY f2 */
    CT_FLAG_KEEP_HITS = 2u,   /* keep the primary-ray hit records for ct_gpu_readback_hits */
    CT_FLAG_COUNT_TESTS = 4u, /* count box / triangle tests (slower; for roofline accounting) */
    CT_FLAG_STAGE_TIMING = 8u, /* bracket every kernel launch of a tile with CUDA events (profiling passes only) */
    CT_FLAG_SUPERSAMPLING = 32u, /* settings.supersampling (raythread.cpp:460-505): 4x4 jittered samples per pixel folded into
                                 the pixel by the reference's running blend.  The reference draws the jitter from libc rand()
                                 on all worker threads at once and is not reproducible; this flag uses a counter-based
                                 generator keyed on (x, y, call number) instead -- the same function the parity
                                 harness substitutes for rand() in the compiled reference (DESIGN.md, sampling modes).  16x the rays of a plain frame.
                                 Combines with CT_FLAG_SUBSAMPLING as in the reference (not with CT_FLAG_KEEP_HITS). */
    CT_FLAG_BUILD_BVH = 64u,  /* ct_gpu_upload_scene builds the tree itself from the triangles (as ct_gpu_build_bvh does, on the device,
                                 in place: nothing goes back to the host); n_nodes must be 0 and nodes, tri_indexes NULL.  A tree deeper
                                 than the device traversal stack is refused with CT_ERR_LIMIT and the previous scene stays loaded */
    CT_FLAG_SUBSAMPLING = 16u /* settings.subsampling (raythread.cpp:512-531): of the rows of a tile (= one worker's
                                 partition) every other one and the last are traced, the rows between get the average
                                 of their neighbours.  Tiles must be rendered in the order the caller wants their
                                 seams resolved (the reference's threads race there); not with ct_gpu_render_shared */
};

/* What RayThread hands its workers (display_partition_t raythread.cpp:69-78 + bvh_state_t bvh.h:19-25). */
typedef struct ct_scene_desc {
    uint32_t struct_size;           /* = sizeof(ct_scene_desc) */
    uint32_t flags;                 /* CT_FLAG_* */

    uint32_t n_triangles;           /* bvh_state_t.triangles.size */
    uint32_t triangle_stride;       /* bytes between triangles: 96 for the reference's triangle_t
                                       (scenefile.h:36-41, 4 x v3_t), 72 for packed p1,p2,p3 */
    const void *triangles;          /* each: 9 doubles p1,p2,p3 at offset 0 (GetSceneTriangles order, raythread.cpp:621) */
    const ct_material *materials;   /* per triangle k: objects[triangleLookup.indexes[k]].material (raythread.cpp:211) */

    uint32_t n_nodes;               /* bvh_state_t.nodesUsed */
    uint32_t n_lights;              /* lightStack.index */
    const ct_bvh_node *nodes;       /* bvh_state_t.bvhNodes, root = node 0 */
    const uint32_t *tri_indexes;    /* bvh_state_t.triangles.indexes (permutation, n_triangles) */
    const ct_light *lights;         /* lightStack.lights, file order (order is part of the result: fp32 accumulation) */

    double camera_position[3];      /* camera_t scenefile.h:68-71 */
    double camera_rotation[9];      /* rotation.data[i][j] row-major (raythread.cpp:564-572) */
    float viewport[3];              /* width,height,d -- the reference always passes {1,1,1} (raythread.cpp:554) */

    int32_t width, height;          /* bitmapSettings_t environment.h:7-12 */
    int32_t max_depth;              /* recursion depth; the reference's literal is 10 (raythread.cpp:508) */
    uint32_t background;            /* 0x333333 (raythread.cpp:59) */
} ct_scene_desc;

/* Rays are counted by kind (SURVEY 8d): primary = pixels traced, shadow = one per non-ambient light
 * per shaded point (raythread.cpp:304), reflection = recursive TraceRay calls (raythread.cpp:373). */
typedef struct ct_ray_counters {
    uint64_t rays_primary, rays_shadow, rays_reflection;
    uint64_t box_tests, tri_tests;  /* only with CT_FLAG_COUNT_TESTS, else 0 */
} ct_ray_counters;

int ct_gpu_abi_version(void);
int ct_gpu_device_count(void);                 /* >= 0, or negative ct_status */
const char *ct_gpu_last_error(void);

/* Replaces RayThread's first-call initialisation hand-off (raythread.cpp:647-654): copies the scene and
 * the BVH built by the reference's BuildBVH (bvh.cpp:108) to `device` as SoA arrays and allocates the
 * device framebuffer (zero-filled, like cobbletrace.cpp:57).  Re-uploading replaces the previous scene. */
int ct_gpu_upload_scene(int device, const ct_scene_desc *desc);

/* The reference's InitializeBVHState + BuildBVH (bvh.cpp:16-120) on `device`: the same tree, node for node and index for
 * index, every field included (_pad = 0), as the reference and ct_host_build_bvh make it.  Triangles are given as in
 * ct_scene_desc: 9 doubles p1,p2,p3 at the start of each record, triangle_stride >= 72 and a multiple of 8.  Writes
 * nodes[0 .. nodesUsed) and tri_indexes[0 .. n_triangles) and returns nodesUsed (= 1 + 2 * interior nodes).
 * nodes_capacity must be at least 2 n - 1 (what InitializeBVHState allocates), else CT_ERR_INVALID; n = 0 is
 * CT_ERR_INVALID, n >= 2^31 CT_ERR_LIMIT.  Trees of any depth are built (the depth limit applies to rendering only).
 * Synchronous; works on a stream and buffers of its own, so a scene uploaded on `device` and its frames are not
 * affected (its kernels may wait for the call: freeing the call's buffers synchronises the device).  A failed allocation
 * returns CT_ERR_OOM and leaves nothing allocated. */
int ct_gpu_build_bvh(int device, uint32_t n_triangles, const void *triangles, uint32_t triangle_stride, ct_bvh_node *nodes,
                     uint32_t nodes_capacity, uint32_t *tri_indexes);

/* What ct_gpu_upload_scene derived from the tree, for tests that compare two uploads (ct_gpu_debug_scene_array "summary"). */
typedef struct ct_scene_summary {
    uint32_t n_pairs;          /* interior nodes (child-pair records) */
    uint32_t n_wide;           /* wide nodes of the early-exit walks (0 for a leaf root) */
    uint32_t root_ref, root_cnt;   /* the root: its pair (interior) or first leaf position and triangle count (leaf) */
    uint32_t pos_of_tri0;      /* leaf position of triangle 0 */
    uint32_t nested;           /* every child box lies inside its parent's */
    uint32_t leaf_dfs_order;   /* leaf positions increase along the reference's DFS */
    uint32_t can_overflow;     /* a walk can exceed the visit budget (parking buffers allocated) */
    double bound[3];           /* largest |coordinate| of any box per axis (INFINITY: some box not finite or unordered) */
    int32_t depth;             /* the tree's depth (DFS stack entries) */
    uint32_t _pad;
} ct_scene_summary;

/* What the frames' path state was sized from, for tests that compare two uploads (ct_gpu_debug_scene_array "path_state"). */
typedef struct ct_path_summary {
    uint32_t n_triangles;
    uint32_t n_lights;
    uint32_t n_shadow_lights;  /* lights that cast shadow rays (all but the ambient ones) */
    uint32_t occ_words;        /* words of occlusion bits per path: ceil(n_lights / 32), at least 1 */
    uint32_t any_leaves;       /* leaf-list entries of the any-hit walk (option "any_leaves" as read at upload, or its rule) */
    uint32_t any_reflective;   /* some material has reflection > 0 or NaN: paths recurse */
    uint32_t levels;           /* path depths the per-depth arrays hold: max_depth + 1 with any_reflective, else 1 */
    uint32_t ovf_cap;          /* rays per parking buffer (0: no walk can be parked, no parking buffers) */
} ct_path_summary;

/* Debug export: copies one of the arrays ct_gpu_upload_scene built into dst and sets *bytes to its size.  Names: "wide",
 * "pairs32", "pairs64", "tris32", "tris", "materials", "pair_parent" (0 bytes when no walk can be parked), "tri_parent",
 * "summary" (a ct_scene_summary), "lights" (the device's light records, file order), "shadow_lights" (the records of the lights
 * that cast shadow rays, file order), "path_state" (a ct_path_summary).  dst == NULL only reports *bytes; capacity < *bytes is
 * CT_ERR_INVALID.  Synchronises. */
int ct_gpu_debug_scene_array(int device, const char *name, void *dst, size_t capacity, size_t *bytes);

/* Replaces the camera half of HandleUpdates (raythread.cpp:557-572) for an already uploaded scene. */
int ct_gpu_set_camera(int device, const double position[3], const double rotation[9]);

/* Optional: launch on the caller's CUDA stream (a cudaStream_t, e.g. torch's current stream) instead of
 * the library's own; pass NULL to go back. */
int ct_gpu_set_stream(int device, void *cuda_stream);

/* Replaces one worker's RayTracePartition pass (raythread.cpp:437-543) over canvas rows
 * y in [y_start, y_end) -- the same half-open range as display_partition_t.yStart/yEnd
 * (raythread.cpp:580-581) -- for all x.  Asynchronous.  If `counters` is non-NULL the call
 * synchronises and returns this tile's ray counts. */
int ct_gpu_render_tile(int device, int y_start, int y_end, ct_ray_counters *counters);

/* ---- one frame on several GPUs (SURVEY 8e) -------------------------------------------------------------------
 * The scene is uploaded to every GPU.  One of them is the ROOT: its framebuffer receives every pixel and it hosts
 * the frame's chunk cursor.  Every GPU renders the SAME tile with ct_gpu_render_shared: its primary-ray warps take
 * chunks of 32 pixels from the root's cursor with atomics over NVLink (dynamic stealing, no host in the loop) and
 * its shading kernels store finished pixels straight into the root's framebuffer (peer stores) -- there is no
 * separate gather step.  The GPUs may be driven by one process or by one process each (CUDA IPC).
 *
 *   root:    ct_gpu_share_export(dev, &h)  -> ship h to the others (it is plain bytes)
 *   others:  ct_gpu_share_attach(dev, &h)
 *   all:     ct_gpu_share_partition(dev, k, n)   (optional, recommended: see below)
 *   frame:   all: ct_gpu_render_shared(dev, y0, y1, ..); ct_gpu_sync(dev); [barrier]; root: ct_gpu_readback(dev, ...)
 * Every participant calls ct_gpu_render_shared once per frame, and nobody starts frame f + 1 before everybody has
 * finished frame f (the barrier).  The root keeps TWO cursors: frame f steals from cursor f & 1 while the root zeroes the
 * other one on its stream, so no reset call and no host synchronisation is needed between frames (ct_gpu_share_reset
 * remains for callers that abandon a frame half way: it zeroes both).
 */
typedef struct ct_gpu_share {
    uint32_t struct_size;            /* = sizeof(ct_gpu_share) */
    int32_t device;                  /* root device index inside the exporting process */
    int64_t pid;                     /* exporting process */
    uint64_t fb_ptr, cursor_ptr;     /* raw device pointers (used when the attaching device is driven by the same process) */
    unsigned char fb_ipc[64], cursor_ipc[64];   /* cudaIpcMemHandle_t of the same two allocations (other processes) */
    int32_t width, height;
    uint64_t frames;                 /* shared frames the root has rendered so far (which of its two cursors comes next) */
} ct_gpu_share;

int ct_gpu_share_export(int device, ct_gpu_share *out);
int ct_gpu_share_attach(int device, const ct_gpu_share *root);   /* root == NULL detaches */
int ct_gpu_share_reset(int device);                              /* root only: zero both cursors; synchronises (not needed in the protocol above) */
/* Declare that `count` GPUs render every shared frame and that this one is number `index` (0..count-1, all different).
 * Then only part of the chunks is stolen: of every 8*count consecutive chunks, 7*count are dealt round-robin
 * (GPU k owns chunks k, k+count, ... -- no remote atomics, and an equal share of the lighting work that follows,
 * which stealing alone does not balance: the GPU next to the cursor steals cheaper and ends up with more paths to
 * light), the last `count` are stolen from the root's cursor as before (absorbs a slower or busier GPU).  Every declared
 * participant must then call ct_gpu_render_shared for every frame.  count <= 1 takes the declaration back: pure stealing,
 * any subset of the GPUs renders the whole frame.  The dealt fraction is option "shared_static_eighths" (0..8, default 7). */
int ct_gpu_share_partition(int device, int index, int count);
/* ct_gpu_render_tile for a frame shared between GPUs.  Without an attach it behaves like a one-GPU frame. */
int ct_gpu_render_shared(int device, int y_start, int y_end, ct_ray_counters *counters);

/* Blocks until all submitted tiles are done, then copies framebuffer rows [row_start,row_end) into
 * dst (bitmap->memory, row stride in pixels).  Only pixels the tracer covers are written: the centred
 * square's columns (all columns with CT_FLAG_WIDE), and never a row the reference never writes
 * (row 0, SURVEY 0.6) -- everything else in dst is left untouched, as the reference leaves it. */
int ct_gpu_readback(int device, uint32_t *dst, int dst_stride_pixels, int row_start, int row_end);

/* The same copy without stalling the renderer, for loops that render frame k + 1 while frame k travels to the host
 * (cobbletrace.cpp:114-118 does RayThread, then Blit, every tick).  ct_gpu_readback_async returns at once: in stream order
 * behind the tiles submitted so far the rows are snapshotted on the device, and a copy stream moves the snapshot into dst
 * -- which should be page-locked (cudaHostAlloc / cudaHostRegister) and must stay valid until ct_gpu_readback_wait(device)
 * has returned.  One copy may be in flight per device; a second request queues behind the first. */
int ct_gpu_readback_async(int device, uint32_t *dst, int dst_stride_pixels, int row_start, int row_end);
int ct_gpu_readback_wait(int device);

/* Debug/parity export (needs CT_FLAG_KEEP_HITS): primary-ray hit records in framebuffer layout.
 * found: 1/0, or 0xFFFFFFFF where no ray was traced.  Any pointer may be NULL. */
int ct_gpu_readback_hits(int device, uint32_t *found, uint32_t *index, float *t, int stride_pixels,
                         int row_start, int row_end);

/* Accumulated counters since upload / last reset (synchronises). */
int ct_gpu_get_counters(int device, ct_ray_counters *out, int reset);

/* Device time in ms spent in the kernels of the most recent ct_gpu_render_tile (CUDA events on the
 * launching stream; synchronises). */
int ct_gpu_last_tile_ms(int device, float *ms);

/* Number of this library's kernels launched on `device` since upload / last reset (the caller's
 * "gpu_launches" claim; memsets and copies are not counted). */
int ct_gpu_kernel_launches(int device, uint64_t *out, int reset);

/* With CT_FLAG_STAGE_TIMING: device time of every kernel of the most recent tile, in launch order.
 * names[i] points at a static string ("primary", "shadow", "shade", "bounce", "overflow_shadow",
 * "overflow_bounce", "resolve"); depth[i] is the path depth.
 * Returns the number of launches (fills at most `max`; a tile never has more than 80). Synchronises. */
int ct_gpu_last_tile_stages(int device, int max, float *ms, const char **names, int *depth);

int ct_gpu_sync(int device);

/* Library-wide tuning knobs, applied by the next ct_gpu_upload_scene.  Names:
 *   "traversal_budget"  node visits + triangle tests a shadow / reflection ray may spend in its own thread
 *                       before it is parked for k_overflow (0 = default 384), which gives it a whole warp and,
 *   "overflow_warp_budget"  after that many node visits (0 = default 4096), hands it to a kernel that tests every triangle
 *                       with the whole grid and checks the ancestor boxes of the ones that pass.
 *                       Results never depend on either; tests set them low to push rays through those paths.
 *   "emulate_ranks"     R > 1: a profiling aid -- every render takes only every R-th chunk of the tile, i.e. the share
 *                       one of R GPUs gets in a shared frame (the other pixels are simply not rendered); applies to
 *                       the next render, 0 / 1 = off.
 *   "shared_static_eighths"  see ct_gpu_share_partition.
 *   "shared_chunk_shift"  log2 of the pixels a warp steals at a time in a shared frame: 5 (default, also 0) or 6.
 *   "primary_budget"    pair visits after which a primary ray's closest-hit walk is given up and the ray parked for a second
 *                       kernel that walks the long rays together (same result; measured slower, DESIGN.md 5): 0 = default (never), < 0 = never.
 *                       Read at upload.
 *   "any_leaves"        leaf-list entries a shadow ray's walk fills before its warp tests the deferred leaves (5..12; larger values mean 12):
 *                       0 = default (12; 8 for scenes with 16 or more shadow-casting lights).  Read at upload.  Never changes a result.
 *   "primary_split"     1: the parked primary rays are finished ONE RAY PER WARP (k_primary_split: the order-free closest-hit search as
 *                       a 32-wide frontier, ~12 rounds instead of up to ~300 dependent visits) instead of 32 rays to a warp; 0 (default).
 *                       Applies to the next render.
 *   "shared_run_shift"  log2 of the run of consecutive 32-pixel chunks (horizontally adjacent 8x4 blocks) that is dealt to /
 *                       stolen by a GPU as one unit in a shared frame: 0 (default) = chunk by chunk.  Every participant of a
 *                       frame must use the same value.
 *   "shadow_reuse"      1 (default): a reflection path whose shading point repeats its parent's (tclosest = 0, see
 *                       ct_gpu_reuse_stats) takes the parent's shadow verdicts instead of tracing the same rays again; 0: trace all.
 *                       Applies to the next render.
 *   "shared_hold_frame" 1: the next ct_gpu_render_shared calls belong to the SAME shared frame as the previous one (same
 *                       cursor, not advanced) -- for tests in which one device plays several participants in turn; 0 = off.
 *   "l2_persist"        1 (default): set aside L2 for persisting lines and open an access-policy window over the walk's
 *                       fp32 records on the render streams; 0: leave the L2 to the default policy (for A/B measurements). */
int ct_gpu_set_option(const char *name, long long value);

/* Rays parked so far on `device` since upload (shadow and reflection rays whose DFS ran past the budget, e.g. the
 * shadow rays of a shading point 2^32 ray lengths away after a reflection miss, SURVEY 0.4), and how many
 * of them found the parking buffer full and were finished by their own thread.  Synchronises. */
int ct_gpu_overflow_stats(int device, uint64_t *parked, uint64_t *finished_in_place);

/* Shadow rays, of those counted in rays_shadow since upload / the last counter reset, that were NOT traced because an
 * ancestor's identical ray had been: the reference builds its reflection rays with t = 0 (raythread.cpp:373), so a reflection
 * "hit" has tclosest = 0 and the next shading point IS the previous one (raythread.cpp:360) -- ComputeLighting casts the
 * same shadow rays again (raythread.cpp:288-304).  Such a path takes its parent's verdicts (option "shadow_reuse", default
 * 1; 0 traces every ray).  Synchronises. */
int ct_gpu_reuse_stats(int device, uint64_t *shadow_rays_reused);

/* With CT_FLAG_COUNT_TESTS: how many of the counted box / triangle tests the certified fp32 filters could not
 * decide and handed to the reference's fp64 arithmetic (since upload / last counter reset).  Synchronises. */
int ct_gpu_filter_stats(int device, uint64_t *box_exact, uint64_t *tri_exact);

/* Blocks until at most `max_in_flight` of the submitted tiles are unfinished (0 == ct_gpu_sync).  Lets a
 * boss keep a GPU fed while tile stealing still follows real progress. */
int ct_gpu_throttle(int device, int max_in_flight);

/* Device framebuffer access for multi-GPU gathers done by the host framework (NCCL / peer copies):
 * pointer to row-major uint32 pixels, stride = width. Valid until the next upload/shutdown. */
int ct_gpu_framebuffer(int device, void **device_ptr, int *width, int *height);

/* In-process multi-GPU gather (north_star "cudaMemcpyPeer" path): copy framebuffer rows
 * [row_start,row_end) of src_device into dst_device's framebuffer over NVLink.  Both devices must hold
 * an uploaded scene of the same frame size.  Asynchronous on src_device's stream. */
int ct_gpu_gather_rows(int src_device, int dst_device, int row_start, int row_end);
/* Rows [row_start, row_end) of `device`'s framebuffer now hold pixels that arrived from outside this library (a
 * collective or peer copy into ct_gpu_framebuffer's pointer): ct_gpu_readback copies only rows known to hold pixels
 * -- those this device rendered, those gathered with ct_gpu_gather_rows, and those marked here. */
int ct_gpu_mark_rows(int device, int row_start, int row_end);

/* ---- ray queries on device memory -----------------------------------------------------------------------------
 * ct_gpu_trace_rays traces n caller rays of one of the three kinds the reference casts through the uploaded scene.  Ray i's
 * outputs equal, bit for bit, what the reference's ClosestIntersection (raythread.cpp:197-227) returns for it:
 *   CT_RAY_PRIMARY     ray.t = 1e30f, the closest hit: found, index (closestIndex: the triangle's id in GetSceneTriangles order,
 *                      0 when none) and tclosest;
 *   CT_RAY_SHADOW      ray.t = 1e30f, occlusion (raythread.cpp:304-306): found = some reachable triangle passes with 1e-4 < t < 1e30;
 *                      index and tclosest are not written;
 *   CT_RAY_REFLECTION  ray.t = 0 (raythread.cpp:373): the first barycentric pass in DFS order; found is always 1, index that
 *                      triangle's id (0 when none), tclosest 0 after a pass and FINF = 2^32 without one.
 * The rays take the walks a frame's rays take, parking and the second-pass kernels included, under the options in effect at
 * upload (traversal_budget, overflow_warp_budget, any_leaves, primary_budget) and at the call (primary_split).
 *
 * Every array lives in DEVICE (or managed) memory of `device` and holds n entries: origins and directions n x 3 doubles (8-byte
 * aligned), found / index / tclosest n entries each (4-byte aligned; each may be NULL).  The call is asynchronous: it enqueues
 * its work on `stream` (NULL = the device's render stream, see ct_gpu_set_stream) and returns; the outputs are valid once the
 * stream reaches that point.  It does not synchronise: its scratch comes from the stream-ordered allocator and is freed in stream
 * order, nothing is kept between calls, and the caller's stream is left as it is (no L2 access-policy window).  Queries read the
 * scene's arrays only: frames, ct_gpu_get_counters, ct_gpu_overflow_stats and ct_gpu_reuse_stats are unchanged by them.  The
 * scene must outlive the queries in flight; ct_gpu_upload_scene and ct_gpu_shutdown release the previous scene with cudaFree,
 * which waits for all work on the device, queries included.
 * Returns CT_OK; CT_ERR_INVALID for a NULL q, a wrong struct_size or kind, NULL rays with n > 0, an array that is not device
 * memory of `device` (host memory, pageable or pinned, is refused) or is misaligned -- all checked before anything is enqueued;
 * CT_ERR_LIMIT for n >= 2^31; CT_ERR_NO_SCENE; CT_ERR_OOM when the scratch cannot be allocated (nothing is enqueued then). */
enum { CT_RAY_PRIMARY = 0, CT_RAY_SHADOW = 1, CT_RAY_REFLECTION = 2 };

typedef struct ct_ray_query {
    uint32_t struct_size;            /* = sizeof(ct_ray_query) */
    int32_t kind;                    /* CT_RAY_* */
    uint32_t n;                      /* rays; 0 is a no-op */
    uint32_t _pad;
    const double *origins;           /* n x 3 doubles, device memory of `device` */
    const double *directions;        /* n x 3 doubles, device memory of `device` */
    uint32_t *found;                 /* n, device memory; each output may be NULL */
    uint32_t *index;                 /* n: closestIndex, 0 when none */
    float *tclosest;                 /* n */
    void *stream;                    /* cudaStream_t to run on; NULL = the device's render stream (ct_gpu_set_stream) */
} ct_ray_query;

int ct_gpu_trace_rays(int device, const ct_ray_query *q);

/* ---- shading queries on device memory -------------------------------------------------------------------------
 * ct_gpu_shade_rays returns, for n caller rays, the colour the reference's TraceRay (raythread.cpp:353-386) returns for them:
 * color[i] = TraceRay({origins[i], directions[i], 1e30f}, 1, FINF, max_depth) as 0x00BBGGRR -- lighting, shadow rays and the
 * reflection recursion included, bit for bit; a ray that hits nothing gets the scene's background.  With no reflective material
 * in the scene the recursion stops at depth 0, as in frames.  The rays go through a frame's own stages (primary, shadow, shade,
 * bounce, ..., resolve) in place of the camera's, so any camera model, sample pattern or batch of views can be shaded.
 * Options apply as they do to frames: traversal_budget, overflow_warp_budget, any_leaves and primary_budget are read at upload,
 * primary_split and shadow_reuse at the call; emulate_ranks and the shared-frame state (ct_gpu_share_*) are ignored -- a query
 * shades every ray on this device.
 *
 * Every array lives in DEVICE (or managed) memory of `device`: origins and directions n x 3 doubles (8-byte aligned), color n
 * words (4-byte aligned).  The call is asynchronous: it enqueues its work on `stream` (NULL = the device's render stream, see
 * ct_gpu_set_stream) and returns; color is valid once the stream reaches that point.  It does not synchronise: its scratch comes
 * from the stream-ordered allocator and is freed in stream order, nothing is kept between calls, and the caller's stream is left
 * as it is (no L2 access-policy window).  The stages run one after the other on that stream (a frame overlaps each depth's
 * lighting with the next depth's hits on side streams the library shares with frames).  Queries read the scene's arrays only:
 * frames, ct_gpu_get_counters, ct_gpu_kernel_launches, ct_gpu_overflow_stats and ct_gpu_reuse_stats are unchanged by them.  The
 * scene must outlive the queries in flight (see ct_gpu_trace_rays).
 *
 * Scratch: the rays are shaded in batches of up to 2^20 that reuse one allocation, so the scratch does not grow with n.  For a
 * batch of B = min(n, 2^20) rays (rounded up to 64), L = max_depth + 1 levels (1 without a reflective material) and the scene's
 * n_lights, counted from the allocation: B x 13 B for L = 1, B x (65 + 76 L) B for L > 1 (hit records, colour and reflection
 * stacks, ray queues with their slot and parent lists, far lists), plus B x L x 4 B x ceil(n_lights / 32) of occlusion words,
 * plus, on a scene whose walks can be parked, 2 x L x 68 B x min(B, the frame's parking capacity: 2^18, or 1/16 of the frame's
 * slots with primary_budget set) of parking buffers -- e.g. about 430 MB at B = 2^20, L = 3, 3 lights.
 * Returns CT_OK; CT_ERR_INVALID for a NULL q, a wrong struct_size, NULL arrays with n > 0, an array that is not device memory of
 * `device` (host memory, pageable or pinned, is refused) or is misaligned; CT_ERR_LIMIT for n >= 2^31 or max_depth > 15;
 * CT_ERR_NO_SCENE -- all checked before anything is enqueued; CT_ERR_OOM when the scratch cannot be allocated (nothing is
 * enqueued then). */
typedef struct ct_shade_query {
    uint32_t struct_size;            /* = sizeof(ct_shade_query) */
    uint32_t n;                      /* rays; 0 is a no-op */
    int32_t max_depth;               /* TraceRay's recursionDepth: 0..15, < 0 = the scene's (as uploaded) */
    uint32_t _pad;
    const double *origins;           /* n x 3 doubles, device memory of `device` */
    const double *directions;        /* n x 3 doubles, device memory of `device` */
    uint32_t *color;                 /* n, device memory: 0x00BBGGRR */
    void *stream;                    /* cudaStream_t to run on; NULL = the device's render stream (ct_gpu_set_stream) */
} ct_shade_query;

int ct_gpu_shade_rays(int device, const ct_shade_query *q);

/* ---- moving a loaded scene's triangles on the device ----------------------------------------------------------------
 * ct_gpu_update_triangles replaces the triangles of the scene loaded on `device` with n_triangles new ones held in device memory
 * -- a mesh deformed or animated on the GPU -- and rebuilds the reference's tree (InitializeBVHState + BuildBVH, bvh.cpp:16-120)
 * over them, on the device, in place.
 *
 * Result: afterwards the device holds exactly the scene ct_gpu_upload_scene with CT_FLAG_BUILD_BVH would load from these triangles
 * plus the scene's current materials, lights, camera, frame size, depth and flags: every array ct_gpu_debug_scene_array exports is
 * equal byte for byte, "summary" included, whether the scene was uploaded with a caller's tree or with the flag (after an update
 * the tree is always BuildBVH's, leaf_dfs_order 1).  Frames and queries that follow equal the reference's on the new triangles.
 *
 * What it keeps -- the update is not an upload: the materials, lights, camera and frame settings; the stream set with
 * ct_gpu_set_stream; a shared-frame attach, partition and frame count (ct_gpu_share_*); the framebuffer, which holds the previous
 * frame's pixels until the next render, and the rows ct_gpu_readback copies; ct_gpu_get_counters, ct_gpu_kernel_launches,
 * ct_gpu_overflow_stats and ct_gpu_reuse_stats.  Options read at upload (traversal_budget, overflow_warp_budget, any_leaves,
 * primary_budget) keep their upload-time values.  ct_gpu_update_scene below also changes the triangle count, materials and lights;
 * this call is its what = CT_UPDATE_TRIANGLES case with the count held fixed.
 *
 * Order: the triangles are read in `stream`'s order (NULL = the render stream, see ct_gpu_set_stream), so work that wrote them on
 * that stream needs no synchronisation by the caller.  The new tree is built into scratch from the stream-ordered allocator first;
 * then the call waits for all work on the device -- frames and queries in flight finish on the old geometry, as they do when a
 * re-upload frees the previous scene -- and overwrites the live arrays, reusing their allocations where the new tree fits.  The
 * call is synchronous: when it returns, `triangles` may be overwritten or freed.  Every participant of a shared frame must update
 * its triangles the same way before the next shared frame; the library does not check this.
 *
 * Returns CT_OK; CT_ERR_INVALID for a NULL u, a wrong struct_size, NULL triangles, n_triangles other than the loaded scene's, a
 * triangle_stride below 72 or not a multiple of 8, triangles that are not device memory of `device` (host memory, pageable or
 * pinned, is refused) or not 8-byte aligned; CT_ERR_NO_SCENE -- all checked before anything is enqueued or changed.  A new tree
 * deeper than the device traversal stack (96) returns CT_ERR_LIMIT and a failed allocation CT_ERR_OOM; in both cases the previous
 * triangles stay loaded and render as before. */
typedef struct ct_triangle_update {
    uint32_t struct_size;            /* = sizeof(ct_triangle_update) */
    uint32_t n_triangles;            /* must equal the loaded scene's */
    uint32_t triangle_stride;        /* as ct_scene_desc: >= 72, a multiple of 8 */
    uint32_t _pad;
    const void *triangles;           /* device memory of `device`: 9 doubles p1,p2,p3 at the start of each record, 8-byte aligned */
    void *stream;                    /* cudaStream_t the triangles are read in the order of; NULL = the render stream */
} ct_triangle_update;

int ct_gpu_update_triangles(int device, const ct_triangle_update *u);

/* ---- editing a loaded scene on the device ---------------------------------------------------------------------------
 * ct_gpu_update_scene replaces any of three parts of the scene loaded on `device` with new ones held in device memory: the
 * triangles (of any count: objects spawned or removed, a tessellation level changed), the materials (an object recoloured) and the
 * lights (a light moved, added or removed) -- geometry, colours and lights generated or animated on the GPU, without a host round trip.
 *
 * Result: afterwards the device holds exactly the scene ct_gpu_upload_scene with CT_FLAG_BUILD_BVH would load from the new parts
 * plus the loaded ones `what` leaves out, with the scene's current camera, frame size, depth, flags, background and viewport, and the
 * options read at upload as they were at upload: every array ct_gpu_debug_scene_array exports is equal byte for byte, "summary",
 * "lights", "shadow_lights" and "path_state" included.  New triangles get BuildBVH's tree (InitializeBVHState + BuildBVH,
 * bvh.cpp:16-120), built on the device; new materials alone or new lights alone leave the tree as it is.  Frames and queries that
 * follow equal the reference's on the edited scene.
 *
 * What it keeps, as ct_gpu_update_triangles does: the camera and frame settings; the stream set with ct_gpu_set_stream; a shared-frame
 * attach, partition and frame count (ct_gpu_share_*); the framebuffer, which holds the previous frame's pixels until the next render,
 * and the rows ct_gpu_readback copies; ct_gpu_get_counters, ct_gpu_kernel_launches, ct_gpu_overflow_stats and ct_gpu_reuse_stats.
 * Frame size, depth and flags do not change: re-upload for those.
 *
 * Order: the inputs are read in `stream`'s order (NULL = the render stream, see ct_gpu_set_stream), so work that wrote them on that
 * stream needs no synchronisation by the caller.  The new state is built into scratch first; then the call waits for all work on the
 * device -- frames and queries in flight finish on the old scene -- and overwrites the live state, reusing each allocation where the
 * new records fit.  The call is synchronous: when it returns, the inputs may be overwritten or freed.  Every participant of a shared
 * frame must apply the same update before the next shared frame; the library does not check this.
 *
 * Returns CT_OK; CT_ERR_INVALID for a NULL u, a wrong struct_size, what == 0 or unknown bits; with CT_UPDATE_TRIANGLES or
 * CT_UPDATE_MATERIALS n_triangles == 0; with CT_UPDATE_TRIANGLES NULL triangles or a triangle_stride below 72 or not a multiple of 8;
 * with CT_UPDATE_MATERIALS NULL materials; a count other than the loaded scene's without both CT_UPDATE_TRIANGLES and
 * CT_UPDATE_MATERIALS (materials are per triangle); with CT_UPDATE_LIGHTS n_lights > 0 and NULL lights; an input that is not device
 * memory of `device` (host memory, pageable or pinned, is refused) or is misaligned (triangles and lights 8 bytes, materials 4);
 * CT_ERR_LIMIT for n_triangles >= 2^31; CT_ERR_NO_SCENE -- all checked before anything is enqueued or changed.  A new tree deeper
 * than the device traversal stack (96) returns CT_ERR_LIMIT and a failed allocation CT_ERR_OOM; in both cases the previous scene
 * stays loaded and renders as before. */
enum { CT_UPDATE_TRIANGLES = 1u, CT_UPDATE_MATERIALS = 2u, CT_UPDATE_LIGHTS = 4u };

typedef struct ct_scene_update {
    uint32_t struct_size;            /* = sizeof(ct_scene_update) */
    uint32_t what;                   /* CT_UPDATE_* mask, != 0 */
    uint32_t n_triangles;            /* CT_UPDATE_TRIANGLES and / or CT_UPDATE_MATERIALS: the new count */
    uint32_t triangle_stride;        /* CT_UPDATE_TRIANGLES: as ct_scene_desc, >= 72, a multiple of 8 */
    uint32_t n_lights;               /* CT_UPDATE_LIGHTS: the new count, 0 allowed (no lights) */
    uint32_t _pad;
    const void *triangles;           /* device memory: 9 doubles p1,p2,p3 at the start of each record, 8-byte aligned */
    const ct_material *materials;    /* device memory: n_triangles records, by triangle id (GetSceneTriangles order), 4-byte aligned */
    const ct_light *lights;          /* device memory: n_lights records, file order, 8-byte aligned (NULL only when n_lights == 0) */
    void *stream;                    /* cudaStream_t the inputs are read in the order of; NULL = the render stream */
} ct_scene_update;

int ct_gpu_update_scene(int device, const ct_scene_update *u);

/* Known-answer-test entry: ClosestIntersection (raythread.cpp:197-227) for n arbitrary rays through the
 * uploaded scene.  origins/directions: n x 3 doubles; t0: initial ray_t.t per ray (1e30f primary/shadow,
 * 0 for the reference's reflection rays, raythread.cpp:373).  Outputs may be NULL. */
int ct_gpu_debug_closest(int device, uint32_t n, const double *origins, const double *directions, const float *t0,
                         uint32_t *found, uint32_t *index, float *tclosest);

/* Known-answer-test entry for the early-exit walks: mode 0 = shadow ray (ray.t = 1e30f, found = occluded, raythread.cpp:304-306),
 * mode 1 = reflection ray (ray.t = 0: index = first barycentric pass in DFS order, 0 when none, raythread.cpp:373).
 * The rays take the path a frame's rays take, with the options in effect at upload (traversal_budget, overflow_warp_budget,
 * any_leaves): the walk, parking, k_overflow, k_overflow_huge.  path[i] (may be NULL): 0 finished by its own walk, 1 by k_overflow,
 * 2 by k_overflow_huge, 3 finished in place (parking buffer full). */
int ct_gpu_debug_early(int device, int mode, uint32_t n, const double *origins, const double *directions,
                       uint32_t *found, uint32_t *index, uint32_t *path);

/* Known-answer-test entry for the primary rays: ClosestIntersection with ray.t = 1e30f (raythread.cpp:197-227) for n arbitrary
 * rays, taking the path a frame's primary rays take under the options in effect at upload (primary_budget) and at the call
 * (primary_split): the walk of k_primary, parking, the real k_primary_long or k_primary_split, or the walk again in place when the
 * parking buffer is full.  park_cap: capacity of the parking buffer, 0 = a frame's (a small value forces the in-place path).
 * found / index / tclosest as ct_gpu_debug_closest returns them.  path[i] (all outputs may be NULL): low byte 0 finished by its own
 * walk, 1 by k_primary_long, 2 by k_primary_split, 3 in place; for 2 the next byte says how k_primary_split decided it: 0 by its
 * frontier and replay, or walked in the reference's order because 1 the ray is outside the rounding analysis (sigma = 0), 2 the tree
 * is not nested, 3 a candidate has t >= FINF, 4 a lane's candidate list is full, 5 the warp's node stack is full, 6 a candidate's
 * leaf box starts beyond the minimum + sigma, 7 more than 32 candidates lie within sigma of the minimum.  Works on buffers of its
 * own: frames rendered afterwards are unchanged. */
int ct_gpu_debug_primary(int device, uint32_t n, const double *origins, const double *directions, uint32_t park_cap,
                         uint32_t *found, uint32_t *index, float *tclosest, uint32_t *path);

/* Known-answer-test entry for the two primitives (bvh.cpp:147 IntersectTriangle, :165 IntersectAABB):
 * n independent (ray, triangle, box) cases.  tri: n x 9, bmin/bmax: n x 3.  ray_t is in/out. */
int ct_gpu_debug_primitives(int device, uint32_t n, const double *origins, const double *directions, float *ray_t,
                            const double *tri, const double *bmin, const double *bmax,
                            uint32_t *tri_hit, uint32_t *box_hit);

/* Soundness test entry for the certified fp32 filters that front IntersectAABB / IntersectTriangle on the device
 * (DESIGN.md 2): n independent (ray, box[, triangle]) cases; tri (n x 9) may be NULL.  The slab filter's per-axis
 * magnitude bound is max(|bmin|,|bmax|) * bound_scale (bound_scale >= 1 imitates a small box inside a large scene).
 * verdict[i]: bit 0 = the reference's box verdict, bits 1-2 = the slab filter's (0 undecided, 1 accept, 2 reject),
 * bit 3 = slab filter usable for this ray, bit 4 = its bracket failed to contain the reference's float tmin/tmax,
 * bit 5 = the division-free fp64 evaluation used for undecided tests differs from the literal arithmetic (4 and 5
 * must never be set); with tri: bit 8 = the reference's IntersectTriangle returns true, bit 9 = ... with
 * 1e-4 < t < 1e30 (what occludes a shadow ray), bit 10 / 11 = the triangle filter says "certainly no effect" for
 * closest-hit / shadow rays (must imply bit 8 / bit 9 clear), bit 12 = triangle filter usable for this ray. */
int ct_gpu_debug_filter(int device, uint32_t n, const double *origins, const double *directions, const float *ray_t,
                        const double *tri, const double *bmin, const double *bmax, double bound_scale, uint32_t *verdict);

/* Known-answer-test entry for the shading arithmetic of ComputeLighting / TraceRay (raythread.cpp:321, :365, :375-379): n
 * independent cases, host arrays, synchronous; no scene is needed.  For each case i, with the functions the frame kernels call:
 *   shaded[i]  = the colour ColorToHsv(color[i]) with v = intensity[i] gives back (HsvToColor), 0x00BBGGRR;
 *   blended[i] = lc[i] * (1 - reflection[i]) + rc[i] * reflection[i] per channel, truncated to uint8_t;
 *   pow_out[i] = pow(x[i], e[i]) in double (the specular term);
 *   acc_out[i] = float(double(acc[i]) + double(li[i]) * pow(x[i], e[i])), the specular accumulation.
 * Any output may be NULL (its inputs may then be NULL too). */
int ct_gpu_debug_shading(int device, uint32_t n, const uint32_t *color, const float *intensity, uint32_t *shaded,
                         const uint32_t *lc, const uint32_t *rc, const float *reflection, uint32_t *blended,
                         const float *x, const int32_t *e, double *pow_out, const float *acc, const float *li, float *acc_out);

/* Frees everything held for `device` (the reference never frees; this makes the library re-entrant). */
int ct_gpu_shutdown(int device);

#ifdef __cplusplus
}
#endif
#endif /* CT_GPU_H */
