/* oracle/ct_oracle.h -- CPU restatement of CobbleTrace's ray/scene intersection +
 * shading path.  TEST INFRASTRUCTURE ONLY: nothing in the product (cobbletrace_b200/,
 * include/) may include, link or call this.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline leg use it, and only as the checker.
 *
 * Parity status: PINNED.  The restatement is checked (tests/test_oracle_vs_ref.py,
 * tests/golden/) against frames, primary-hit maps and BVH dumps produced by the
 * unmodified reference compiled under oracle/_ref (recipe: oracle/Makefile), which in
 * turn reproduces the four 640x640 frame hashes recorded in SURVEY.md 8(c).
 *
 * All file:line citations are relative to /root/reference.
 */
#ifndef CT_ORACLE_H
#define CT_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* lightType_t order, scenefile.h:13 */
enum { CT_ORACLE_LT_POINT = 0, CT_ORACLE_LT_DIRECTIONAL = 1, CT_ORACLE_LT_AMBIENT = 2 };

/* Flattened scene: what RayThread's first call derives from scene_t (raythread.cpp:647-654)
 * plus the arrays ComputeLighting/TraceRay read.  All pointers are borrowed. */
typedef struct ct_oracle_scene {
    uint32_t n_tri, n_lights, n_nodes, _pad;
    const double *tri;              /* n_tri x 9: p1,p2,p3 (triangle_t scenefile.h:36-41) */
    const uint32_t *mat_color;      /* material_t scenefile.h:25-29, per triangle via triangleLookup */
    const int32_t *mat_specular;
    const float *mat_reflection;
    const int32_t *light_type;      /* light_t scenefile.h:61-66, file order */
    const float *light_intensity;
    const double *light_pos;        /* n_lights x 3 */
    const double *light_dir;        /* n_lights x 3 */
    double cam_pos[3];              /* camera_t scenefile.h:68-71 */
    double cam_rot[9];              /* rotation.data[i][j] row-major */
    const double *node_min;         /* bvh_node_t bvh.h:5-11, n_nodes x 3 */
    const double *node_max;
    const uint32_t *node_left, *node_first, *node_count;
    const uint32_t *tri_index;      /* bvh_triangles_t.indexes bvh.h:16 */
} ct_oracle_scene;

typedef struct ct_oracle_counters {
    uint64_t rays_primary, rays_shadow, rays_reflection;
    uint64_t box_tests, tri_tests;  /* IntersectAABB / IntersectTriangle calls, all rays */
    uint64_t box_tests_kind[3], tri_tests_kind[3];  /* the same split by ray kind: 0 primary, 1 shadow, 2 reflection */
    uint64_t ray_hist[3][32];       /* rays by floor(log2(box tests of the ray)), per kind: the traversal-length tail */
    uint64_t box_hist[3][32];       /* box tests spent in each of those buckets */
} ct_oracle_counters;

typedef struct ct_oracle_hit { uint32_t found, index; float t; } ct_oracle_hit;

enum {
    CT_ORACLE_WIDE = 1,     /* trace x in [-W/2, W/2) instead of the reference's centred square (SURVEY f2) */
    CT_ORACLE_SUPERSAMPLE = 4, /* settings.supersampling (raythread.cpp:460-505): 4x4 jittered samples per pixel, running blend; the
                               jitter comes from a counter-based generator instead of rand() (oracle/ref_driver.cpp CT_RAND) */
    CT_ORACLE_SUBSAMPLE = 2 /* settings.subsampling (raythread.cpp:512-531): every other row of [y_start,y_end) is traced, the
                               rows between are averages; each thread's row range is one partition (use n_threads = 1) */
};

/* BVH build, bvh.cpp:16-120.  Arrays sized: node_* for 2*n_tri-1 nodes, tri_index n_tri. Returns nodesUsed. */
uint32_t ct_oracle_build_bvh(uint32_t n_tri, const double *tri, double *node_min, double *node_max,
                             uint32_t *node_left, uint32_t *node_first, uint32_t *node_count, uint32_t *tri_index);

/* Camera matrix, raythread.cpp:564-572 */
void ct_oracle_camera_rotation(float yaw, float pitch, float roll, double out[9]);

/* Pixel loop of RayTracePartition (raythread.cpp:452-537, non-sampled branch) for canvas rows
 * y in [y_start, y_end).  frame: W*H uint32 (only traced pixels are written).  hits (optional): W*H
 * records for the primary rays (found = 0xFFFFFFFF where nothing was stored).  counters optional.
 * n_threads >= 1 splits rows statically.  Returns 0. */
int ct_oracle_render(const ct_oracle_scene *s, int W, int H, int y_start, int y_end, int max_depth, int flags,
                     uint32_t *frame, ct_oracle_hit *hits, ct_oracle_counters *counters, int n_threads);

/* Single-call entry points for known-answer tests. */
int ct_oracle_intersect_triangle(const double org[3], const double dir[3], float *ray_t, const double tri[9]); /* bvh.cpp:147 */
int ct_oracle_intersect_aabb(const double org[3], const double dir[3], float ray_t, const double bmin[3], const double bmax[3]); /* bvh.cpp:165 */
/* ClosestIntersection (raythread.cpp:197-227) for an arbitrary ray; returns found, fills index/t. */
int ct_oracle_closest(const ct_oracle_scene *s, const double org[3], const double dir[3], float ray_t0,
                      uint32_t *index, float *tclosest);
/* ct_oracle_closest for n rays (org / dir: n x 3, ray_t0[n]); found, index, tclosest: n each. */
void ct_oracle_closest_many(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, const float *ray_t0,
                            uint32_t *found, uint32_t *index, float *tclosest);
uint32_t ct_oracle_shade_color(uint32_t material_color, float intensity); /* ColorToHsv + HsvToColor, color.h:114-126 */
uint32_t ct_oracle_blend(uint32_t local_color, uint32_t reflected_color, float reflection); /* raythread.cpp:375-379 */

/* Prototype of the order-free pre-hit phase of a closest-hit walk (see the comment in ct_oracle.c): must agree with
 * ct_oracle_closest for ray_t0 = 1e30.  Tables: node_parent[n_nodes], leaf_of_pos[n_tri]. */
void ct_oracle_prehit_tables(const ct_oracle_scene *s, uint32_t *node_parent, uint32_t *leaf_of_pos);
int ct_oracle_closest_prehit(const ct_oracle_scene *s, const uint32_t *node_parent, const uint32_t *leaf_of_pos,
                             const double org[3], const double dir[3], uint32_t *index, float *tclosest);
/* Both walks over n rays; returns how many differ in found / index / tclosest (bitwise). */
uint64_t ct_oracle_prehit_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, uint64_t *n_found);

/* Prototype of the order-free closest-hit walk (see the comment in ct_oracle.c).  order: 0 left child first, 1 nearer child first.
 * Returns found, or -1 where the ordered walk must decide.  stats[4]: box tests, triangle tests, fallbacks, max candidates. */
int ct_oracle_closest_free(const ct_oracle_scene *s, const double org[3], const double dir[3], int order,
                           uint32_t *index, float *tclosest, uint64_t *stats);
uint64_t ct_oracle_free_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, int order,
                              uint64_t *stats, uint64_t *ref_stats);

/* Prototype of ONE walk split across a warp: the order-free search as a frontier of up to 32 nodes per round (ct_oracle.c). */
int ct_oracle_closest_rounds(const ct_oracle_scene *s, const double org[3], const double dir[3], uint32_t *index, float *tclosest,
                             uint32_t *rounds, uint32_t *pair_visits);
void ct_oracle_rounds_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, uint32_t min_visits, uint64_t out[8]);

/* The slop bound of the order-free walk, measured on (ray, triangle) cases: out[0] passes, out[1] max (tmin(box) - t) / M, out[2] skipped. */
void ct_oracle_slop_check(uint64_t n, const double *org, const double *dir, const double *tri, double out[3]);

#ifdef __cplusplus
}
#endif
#endif
