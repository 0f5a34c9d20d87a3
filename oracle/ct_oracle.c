/* oracle/ct_oracle.c -- plain-C CPU restatement of CobbleTrace's per-pixel ray/scene
 * intersection + shading path.  TEST INFRASTRUCTURE ONLY (see ct_oracle.h): the product
 * never links or calls this.  Parity: PINNED against oracle/_ref (the compiled reference).
 *
 * The reference's arithmetic is mixed (SURVEY 0.2): v3_t is double (mymath.h:24-28) but
 * DotProduct / Magnitude / V3ByIndex return float (mymath.h:229,213,179) and most scalars
 * of the hot path are float.  Every such rounding point is written out explicitly below as
 * a (float) cast of a double expression.  Build with -ffp-contract=off, no -ffast-math.
 *
 * Citations are file:line in /root/reference.
 */
#include "ct_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#define RAY_T_INIT 1e30f            /* ray_t.t of primary and shadow rays, raythread.cpp:508,304 */
static const float FINF = 4294967296.0f;          /* raythread.cpp:58 */
#define BACKGROUND 0x333333u        /* raythread.cpp:59 */

/* mymath.h:11-17 -- macros, NOT fminf/fmaxf: with a NaN operand the comparison is false
 * and the SECOND operand is returned. */
#define MACRO_MIN(a, b) (((a) < (b)) ? (a) : (b))
#define MACRO_MAX(a, b) (((a) > (b)) ? (a) : (b))

typedef struct { double x, y, z; } vec3;

static inline vec3 v_sub(vec3 a, vec3 b) { vec3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }   /* mymath.h:147 */
static inline vec3 v_add(vec3 a, vec3 b) { vec3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }   /* mymath.h:129 */
static inline vec3 v_scale(double s, vec3 a) { vec3 r = {s * a.x, s * a.y, s * a.z}; return r; }     /* mymath.h:47 */
static inline vec3 v_neg(vec3 a) { vec3 r = {-a.x, -a.y, -a.z}; return r; }                          /* mymath.h:118 */
static inline vec3 v_cross(vec3 a, vec3 b) {                                                         /* mymath.h:234 */
    vec3 r = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
    return r;
}
/* mymath.h:229 -- double sum, left to right, rounded to float on return */
static inline float v_dot(vec3 a, vec3 b) { return (float)(a.x * b.x + a.y * b.y + a.z * b.z); }
/* mymath.h:213 -- double sqrt, rounded to float on return */
static inline float v_mag(vec3 a) { return (float)sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }
static inline vec3 v_load(const double *p) { vec3 r = {p[0], p[1], p[2]}; return r; }

typedef struct { vec3 org, dir; float t; } ray;   /* ray_t, scenefile.h:104-108 */

typedef struct {
    const ct_oracle_scene *s;
    ct_oracle_counters c;
    int kind;               /* kind of the ray being traversed: 0 primary, 1 shadow, 2 reflection */
} ctx;

/* ---- bvh.cpp:147-163 IntersectTriangle -------------------------------------------- */
static int intersect_triangle(ray *r, const double *tri) {
    vec3 p1 = v_load(tri), p2 = v_load(tri + 3), p3 = v_load(tri + 6);
    vec3 edge1 = v_sub(p2, p1);
    vec3 edge2 = v_sub(p3, p1);
    vec3 h = v_cross(r->dir, edge2);
    float a = v_dot(edge1, h);
    if (a > -0.0001f && a < 0.0001f) return 0;
    float f = 1 / a;
    vec3 sv = v_sub(r->org, p1);
    float u = f * v_dot(sv, h);
    if (u < 0 || u > 1) return 0;
    vec3 q = v_cross(sv, edge1);
    float v = f * v_dot(r->dir, q);
    if (v < 0 || u + v > 1) return 0;
    float t = f * v_dot(edge2, q);
    if (t > 0.0001f) r->t = MACRO_MIN(r->t, t);
    return 1;   /* true whatever the sign/size of t (SURVEY 0.4) */
}

/* ---- bvh.cpp:165-179 IntersectAABB -------------------------------------------------- */
static int intersect_aabb(const ray *r, const double *bmin, const double *bmax) {
    float tx1 = (float)((bmin[0] - r->org.x) / r->dir.x);
    float tx2 = (float)((bmax[0] - r->org.x) / r->dir.x);
    float tmin = MACRO_MIN(tx1, tx2);
    float tmax = MACRO_MAX(tx1, tx2);
    float ty1 = (float)((bmin[1] - r->org.y) / r->dir.y);
    float ty2 = (float)((bmax[1] - r->org.y) / r->dir.y);
    tmin = MACRO_MAX(tmin, MACRO_MIN(ty1, ty2));
    tmax = MACRO_MIN(tmax, MACRO_MAX(ty1, ty2));
    float tz1 = (float)((bmin[2] - r->org.z) / r->dir.z);
    float tz2 = (float)((bmax[2] - r->org.z) / r->dir.z);
    tmin = MACRO_MAX(tmin, MACRO_MIN(tz1, tz2));
    tmax = MACRO_MIN(tmax, MACRO_MAX(tz1, tz2));
    return tmax >= tmin && tmin < r->t && tmax > 0;
}

/* ---- bvh.cpp:198-222 IntersectBVHClosest (recursive, left child first, no ordering) -- */
static void bvh_closest(ctx *cx, ray *r, uint32_t node, float *tclosest, uint32_t *closest_index) {
    const ct_oracle_scene *s = cx->s;
    cx->c.box_tests++;
    cx->c.box_tests_kind[cx->kind]++;
    if (!intersect_aabb(r, s->node_min + 3 * (size_t)node, s->node_max + 3 * (size_t)node)) return;
    uint32_t count = s->node_count[node];
    if (count > 0) {
        uint32_t first = s->node_first[node];
        for (uint32_t i = 0; i < count; i++) {
            uint32_t k = s->tri_index[first + i];
            cx->c.tri_tests++;
            cx->c.tri_tests_kind[cx->kind]++;
            int hit = intersect_triangle(r, s->tri + 9 * (size_t)k);
            if (hit && r->t != RAY_T_INIT && r->t < *tclosest) {
                *closest_index = k;
                *tclosest = r->t;
            }
        }
    } else {
        bvh_closest(cx, r, s->node_left[node], tclosest, closest_index);
        bvh_closest(cx, r, s->node_left[node] + 1, tclosest, closest_index);
    }
}

/* ---- raythread.cpp:197-227 ClosestIntersection (tmin/tmax are ignored there too) ------ */
static int closest_intersection(ctx *cx, ray r, float *tclosest, uint32_t *closest_index) {
    *tclosest = FINF;
    *closest_index = 0;
    uint64_t before = cx->c.box_tests;
    bvh_closest(cx, &r, 0, tclosest, closest_index);
    uint64_t n = cx->c.box_tests - before;
    int b = 0;
    while ((n >> (b + 1)) != 0 && b < 31) b++;
    cx->c.ray_hist[cx->kind][b]++;
    cx->c.box_hist[cx->kind][b] += n;
    return r.t != RAY_T_INIT;
}

/* ---- raythread.cpp:270-273 ReflectRay: 2.0*normal*Dot(normal,ray) - ray ---------------- */
static vec3 reflect_ray(vec3 rv, vec3 normal) {
    double d = (double)v_dot(normal, rv);
    vec3 two_n = v_scale(2.0, normal);
    return v_sub(v_scale(d, two_n), rv);
}

/* ---- raythread.cpp:275-327 ComputeLighting --------------------------------------------- */
static float compute_lighting(ctx *cx, vec3 position, vec3 normal, vec3 view, int specular) {
    const ct_oracle_scene *s = cx->s;
    float intensity = 0.0f;
    for (uint32_t i = 0; i < s->n_lights; i++) {
        float li = s->light_intensity[i];
        vec3 light_ray;
        switch (s->light_type[i]) {
        case CT_ORACLE_LT_AMBIENT:
            intensity += li;
            continue;
        case CT_ORACLE_LT_POINT:
            light_ray = v_sub(v_load(s->light_pos + 3 * i), position);
            break;
        default: /* directional */
            light_ray = v_load(s->light_dir + 3 * i);
            break;
        }
        /* shadow check :304 -- full closest traversal from the surface point, no offset, no t<=1 test */
        ray sr = {position, light_ray, RAY_T_INIT};
        float tc; uint32_t idx;
        cx->c.rays_shadow++;
        int kind_saved = cx->kind;
        cx->kind = 1;
        int shadowed = closest_intersection(cx, sr, &tc, &idx);
        cx->kind = kind_saved;
        if (shadowed) continue;

        float n_dot_l = v_dot(normal, light_ray);                       /* :310 */
        if (n_dot_l > 0) intensity += li * n_dot_l / (v_mag(normal) * v_mag(light_ray));   /* all float :312 */

        if (specular != -1) {                                           /* :316 */
            vec3 refl = reflect_ray(light_ray, normal);
            float r_dot_v = v_dot(refl, view);
            if (r_dot_v > 0) {
                /* :320-321  pow(float,int) is the double pow; the product is double and the
                 * += rounds (double)intensity + product back to float. */
                float q = r_dot_v / (v_mag(refl) * v_mag(view));
                intensity = (float)((double)intensity + (double)li * pow((double)q, (double)specular));
            }
        }
    }
    return intensity;
}

/* ---- color.h ------------------------------------------------------------------------------ */
typedef struct { float h, s, v; } hsv;

static hsv color_to_hsv(uint32_t color) {      /* color.h:114-120 + RgbToHsv :49-75 */
    float r = (float)(color & 0xff) / 0xff, g = (float)((color >> 8) & 0xff) / 0xff, b = (float)((color >> 16) & 0xff) / 0xff;
    float gb_max = MACRO_MAX(g, b), gb_min = MACRO_MIN(g, b);
    float max_c = MACRO_MAX(r, gb_max);
    float min_c = MACRO_MIN(r, gb_min);
    float delta = max_c - min_c;
    hsv o;
    o.v = max_c;
    if (max_c != 0.0) {
        o.s = delta / max_c;
    } else {
        o.s = 0.0f; o.h = -1; return o;
    }
    if (r == max_c) o.h = (g - b) / delta;
    else if (g == max_c) o.h = 2 + (b - r) / delta;
    else o.h = 4 + (r - g) / delta;
    o.h = (float)((double)o.h * 60.0);
    if (o.h < 0) o.h = (float)((double)o.h + 360.0);
    return o;
}

static uint8_t to_u8(float x) { return (uint8_t)(int)x; }   /* float -> uint8_t argument conversion (truncation) */

static uint32_t hsv_to_color(hsv c) {          /* color.h:122-126 + HsvToRgb :18-45 */
    float r, g, b;
    if (c.s == 0) {
        r = g = b = c.v;
    } else {
        c.h = (float)((double)c.h / 60.0);
        int i = (int)floor((double)c.h);
        float f = c.h - i;
        float aa = c.v * (1 - c.s);
        float bb = c.v * (1 - (c.s * f));
        float cc = c.v * (1 - (c.s * (1 - f)));
        r = g = b = 0; /* the reference leaves them uninitialised for i outside 0..5 (color.h:35-42) */
        switch (i) {
        case 0: r = c.v; g = cc;  b = aa;  break;
        case 1: r = bb;  g = c.v; b = aa;  break;
        case 2: r = aa;  g = c.v; b = cc;  break;
        case 3: r = aa;  g = bb;  b = c.v; break;
        case 4: r = cc;  g = aa;  b = c.v; break;
        case 5: r = c.v; g = aa;  b = bb;  break;
        }
    }
    float r255 = r * 0xff, g255 = g * 0xff, b255 = b * 0xff;
    uint8_t R = to_u8(MACRO_MIN(r255, 0xff)), G = to_u8(MACRO_MIN(g255, 0xff)), B = to_u8(MACRO_MIN(b255, 0xff));
    return ((uint32_t)B << 16) | ((uint32_t)G << 8) | R;     /* 0x00BBGGRR color.h:77-80 */
}

uint32_t ct_oracle_shade_color(uint32_t material_color, float intensity) {
    hsv c = color_to_hsv(material_color);
    c.v = intensity;                              /* raythread.cpp:365 */
    return hsv_to_color(c);
}

/* raythread.cpp:375-379: per channel local*(1-r) + reflected*r in double, truncated to uint8_t */
uint32_t ct_oracle_blend(uint32_t lc, uint32_t rc, float reflection) {
    double wl = (double)(1 - reflection), wr = (double)reflection;
    uint32_t out = 0;
    for (int sh = 0; sh <= 16; sh += 8) {
        double l = (double)((lc >> sh) & 0xff), r = (double)((rc >> sh) & 0xff);
        double c = wl * l + wr * r;
        out |= (uint32_t)(uint8_t)(int)c << sh;
    }
    return out;
}

/* ---- raythread.cpp:353-386 TraceRay ------------------------------------------------------------ */
static uint32_t trace_ray(ctx *cx, ray r, int depth) {
    const ct_oracle_scene *s = cx->s;
    float tclosest; uint32_t idx;
    if (!closest_intersection(cx, r, &tclosest, &idx)) return BACKGROUND;
    const double *tri = s->tri + 9 * (size_t)idx;
    vec3 position = v_add(r.org, v_scale((double)tclosest, r.dir));                 /* :360 */
    /* NormalOfSceneObject :336-346: raw cross product, flipped to face the viewer */
    vec3 n = v_cross(v_sub(v_load(tri + 3), v_load(tri)), v_sub(v_load(tri + 6), v_load(tri)));
    float d = v_dot(n, r.dir);
    vec3 normal = (d < 0) ? n : v_neg(n);
    float intensity = compute_lighting(cx, position, normal, v_neg(r.dir), s->mat_specular[idx]);
    uint32_t local = ct_oracle_shade_color(s->mat_color[idx], intensity);
    float reflection = s->mat_reflection[idx];
    if (depth <= 0 || reflection <= 0) return local;                                 /* :369 */
    vec3 rdir = reflect_ray(v_neg(r.dir), normal);                                   /* :372 */
    ray rr = {position, rdir, 0.0f};                                                 /* :373 -- t = 0 (sic) */
    cx->c.rays_reflection++;
    cx->kind = 2;
    uint32_t reflected = trace_ray(cx, rr, depth - 1);
    return ct_oracle_blend(local, reflected, reflection);
}

/* ---- pixel loop, raythread.cpp:452-510 + CanvasToViewport :186-194 + CanvasPutPixel :176-184 --- */
typedef struct {
    ctx cx;
    int W, H, y0, y1, max_depth, flags;
    uint32_t *frame;
    ct_oracle_hit *hits;
} job;

/* The counter-based stand-in for rand() in the supersampling jitter (see oracle/ref_driver.cpp CT_RAND): keyed on the
 * pixel and the number of the call inside it. */
static uint32_t hash3(uint32_t x, uint32_t y, uint32_t k) {
    uint32_t h = x * 0x9E3779B1u ^ (y * 0x85EBCA77u) ^ (k * 0xC2B2AE3Du);
    h ^= h >> 16; h *= 0x7FEB352Du; h ^= h >> 15; h *= 0x846CA68Bu; h ^= h >> 16;
    return h;
}

/* One primary ray through canvas point (px, py) (floats, as the reference passes them): CanvasToViewport :186-194
 * times the camera matrix (mymath.h:68-75), then TraceRay. */
static uint32_t trace_canvas_point(job *j, float px, float py, int want_hit, int stored, int row, int col) {
    const ct_oracle_scene *s = j->cx.s;
    float sx = 1.0f / (float)j->H, sy = 1.0f / (float)j->H;   /* :189-192 viewport {1,1,1} :554, float quotient */
    const double *m = s->cam_rot;
    double vx = (double)px * (double)sx, vy = (double)py * (double)sy, vz = 1.0;
    vec3 dir;                                  /* v3_t * m3x3_t, mymath.h:68-75 */
    dir.x = vx * m[0] + vy * m[3] + vz * m[6];
    dir.y = vx * m[1] + vy * m[4] + vz * m[7];
    dir.z = vx * m[2] + vy * m[5] + vz * m[8];
    ray r = {v_load(s->cam_pos), dir, RAY_T_INIT};
    j->cx.c.rays_primary++;
    if (want_hit && j->hits && stored) {
        ctx tmp; memset(&tmp, 0, sizeof tmp); tmp.s = s;
        ct_oracle_hit *h = &j->hits[(size_t)row * j->W + col];
        h->found = (uint32_t)closest_intersection(&tmp, r, &h->t, &h->index);
    }
    j->cx.kind = 0;
    return trace_ray(&j->cx, r, j->max_depth);
}

static void *render_rows(void *arg) {
    job *j = (job *)arg;
    int W = j->W, H = j->H;
    float half = (float)(H / 2);                 /* :454 float width = bitmap->height/2 (int division) */
    int x_lo = (int)-half, x_hi = (int)half;
    if (j->flags & CT_ORACLE_WIDE) { x_lo = -(W / 2); x_hi = W - W / 2; }
    const int subsample = (j->flags & CT_ORACLE_SUBSAMPLE) != 0, supersample = (j->flags & CT_ORACLE_SUPERSAMPLE) != 0;
    for (int x = x_lo; x < x_hi; x++) {
        uint32_t last_color = 0;                       /* :456 */
        for (int y = j->y0; y < j->y1;) {              /* :457 -- the increment depends on settings.subsampling */
            int col = x + W / 2, row = H / 2 - y;      /* :181-182 */
            int stored = !(row < 0 || row >= H || col < 0 || col >= W);   /* draw2d.h:11-14 */
            uint32_t color = 0;
            if (supersample) {                         /* :460-505, rand() -> hash3(x, y, call number) */
                const int samples = 4;
                float denom = samples * 2;
                float stepsize = 1 / (float)samples;
                float jitter = stepsize / 8;
                float sampleX = (float)x;
                int first = 1;
                uint32_t call = 0;
                for (int xs = 0; xs < samples; xs++) {
                    float sampleY = (float)y;
                    for (int ys = 0; ys < samples; ys++) {
                        float rx = (float)(int)(hash3((uint32_t)x, (uint32_t)y, call++) & 0x7FFFFFFFu) / (float)2147483647;
                        float ry = (float)(int)(hash3((uint32_t)x, (uint32_t)y, call++) & 0x7FFFFFFFu) / (float)2147483647;
                        rx = (rx * (2 * jitter)) - jitter;
                        ry = (ry * (2 * jitter)) - jitter;
                        sampleX += rx;
                        sampleY += ry;
                        uint32_t temp = trace_canvas_point(j, sampleX, sampleY, 0, stored, row, col);
                        if (first) {
                            first = 0;
                            color = temp;
                        } else {                       /* :486-497: running blend in float rgb, truncated to uint8 each time */
                            uint32_t out = 0;
                            for (int sh = 0; sh <= 16; sh += 8) {
                                float c = (float)((color >> sh) & 0xffu), t = (float)((temp >> sh) & 0xffu);
                                c -= (c / denom);
                                c += (t / denom);
                                out |= (uint32_t)(unsigned char)c << sh;
                            }
                            color = out;
                        }
                        sampleY -= ry;
                        sampleY += stepsize;
                        sampleX -= rx;
                    }
                    sampleX += stepsize;
                }
            } else {
                color = trace_canvas_point(j, (float)x, (float)y, 1, stored, row, col);
            }
            if (stored) j->frame[(size_t)row * W + col] = color;
            if (subsample) {                           /* :512-531 */
                if (y == j->y0) last_color = color;
                /* rgb_t holds floats (color.h:11-13): (a + b)/2 in float, min with 0xff, truncated by the uint8_t
                 * parameters of RgbToColor (color.h:77-85) */
                uint32_t avg = 0;
                for (int sh = 0; sh <= 16; sh += 8) {
                    float a = (float)((last_color >> sh) & 0xffu), b = (float)((color >> sh) & 0xffu);
                    float m = (a + b) / 2;
                    m = MACRO_MIN(m, (float)0xff);
                    avg |= (uint32_t)(unsigned char)m << sh;
                }
                int row2 = H / 2 - (y - 1);            /* CanvasPutPixel(bitmap, {x, y-1}, avgColor) */
                if (!(row2 < 0 || row2 >= H || col < 0 || col >= W)) j->frame[(size_t)row2 * W + col] = avg;
                if (y + 2 >= j->y1) y++; else y += 2;
            } else {
                y++;
            }
            last_color = color;
        }
    }
    return NULL;
}

int ct_oracle_render(const ct_oracle_scene *s, int W, int H, int y_start, int y_end, int max_depth, int flags,
                     uint32_t *frame, ct_oracle_hit *hits, ct_oracle_counters *counters, int n_threads) {
    if (n_threads < 1) n_threads = 1;
    int rows = y_end - y_start;
    if (rows <= 0) return 0;
    if (n_threads > rows) n_threads = rows;
    if (hits) for (size_t i = 0; i < (size_t)W * H; i++) if (0) hits[i].found = 0; /* caller pre-fills */
    job *jobs = (job *)calloc((size_t)n_threads, sizeof(job));
    pthread_t *th = (pthread_t *)calloc((size_t)n_threads, sizeof(pthread_t));
    for (int i = 0; i < n_threads; i++) {
        jobs[i].cx.s = s;
        jobs[i].W = W; jobs[i].H = H; jobs[i].max_depth = max_depth; jobs[i].flags = flags;
        jobs[i].y0 = y_start + (int)((long long)rows * i / n_threads);
        jobs[i].y1 = y_start + (int)((long long)rows * (i + 1) / n_threads);
        jobs[i].frame = frame; jobs[i].hits = hits;
        if (n_threads == 1) render_rows(&jobs[i]);
        else pthread_create(&th[i], NULL, render_rows, &jobs[i]);
    }
    ct_oracle_counters total; memset(&total, 0, sizeof total);
    for (int i = 0; i < n_threads; i++) {
        if (n_threads > 1) pthread_join(th[i], NULL);
        total.rays_primary += jobs[i].cx.c.rays_primary;
        total.rays_shadow += jobs[i].cx.c.rays_shadow;
        total.rays_reflection += jobs[i].cx.c.rays_reflection;
        total.box_tests += jobs[i].cx.c.box_tests;
        total.tri_tests += jobs[i].cx.c.tri_tests;
        for (int k = 0; k < 3; k++) {
            total.box_tests_kind[k] += jobs[i].cx.c.box_tests_kind[k];
            total.tri_tests_kind[k] += jobs[i].cx.c.tri_tests_kind[k];
            for (int b = 0; b < 32; b++) {
                total.ray_hist[k][b] += jobs[i].cx.c.ray_hist[k][b];
                total.box_hist[k][b] += jobs[i].cx.c.box_hist[k][b];
            }
        }
    }
    if (counters) *counters = total;
    free(jobs); free(th);
    return 0;
}

/* ---- raythread.cpp:564-572 camera matrix.  The angles are float and <math.h> is the C++ wrapper there, so
 * cos/sin are the float overloads and the arithmetic is fp32 (checked against oracle/_ref --keys). -------- */
void ct_oracle_camera_rotation(float yaw, float pitch, float roll, double o[9]) {
    float cy = cosf(yaw), sy = sinf(yaw), cp = cosf(pitch), sp = sinf(pitch), cr = cosf(roll), sr = sinf(roll);
    o[0] = (double)(cy * cp);  o[1] = (double)(cy * sp * sr - sy * cr);  o[2] = (double)(cy * sp * cr + sy * sr);
    o[3] = (double)(sy * cp);  o[4] = (double)(sy * sp * sr + cy * cr);  o[5] = (double)(sy * sp * cr - cy * sr);
    o[6] = (double)(-sy);      o[7] = (double)(cp * sr);                 o[8] = (double)(cp * cr);
}

/* ---- single-call KAT entry points ------------------------------------------------------------------- */
int ct_oracle_intersect_triangle(const double org[3], const double dir[3], float *ray_t, const double tri[9]) {
    ray r = {v_load(org), v_load(dir), *ray_t};
    int hit = intersect_triangle(&r, tri);
    *ray_t = r.t;
    return hit;
}

int ct_oracle_intersect_aabb(const double org[3], const double dir[3], float ray_t, const double bmin[3], const double bmax[3]) {
    ray r = {v_load(org), v_load(dir), ray_t};
    return intersect_aabb(&r, bmin, bmax);
}

int ct_oracle_closest(const ct_oracle_scene *s, const double org[3], const double dir[3], float ray_t0,
                      uint32_t *index, float *tclosest) {
    ctx cx; memset(&cx, 0, sizeof cx); cx.s = s;
    ray r = {v_load(org), v_load(dir), ray_t0};
    *tclosest = FINF;
    *index = 0;
    bvh_closest(&cx, &r, 0, tclosest, index);
    return r.t != RAY_T_INIT;
}

void ct_oracle_closest_many(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, const float *ray_t0,
                            uint32_t *found, uint32_t *index, float *tclosest) {
    for (uint64_t i = 0; i < n; i++)
        found[i] = (uint32_t)ct_oracle_closest(s, org + 3 * i, dir + 3 * i, ray_t0[i], index + i, tclosest + i);
}

/* ---- bvh.cpp:16-120 build: midpoint split on the longest axis, leaves <= 2 or unsplittable -------- */
typedef struct {
    uint32_t n_tri, used;
    const double *tri;
    double *centroid;       /* n_tri x 3, BuildBVH :112 */
    double *nmin, *nmax;
    uint32_t *left, *first, *count, *index;
} builder;

static inline float by_axis_f(const double *v, int axis) { return (float)v[axis]; }   /* V3ByIndex mymath.h:179 returns float */

static void update_bounds(builder *b, uint32_t node) {                                   /* bvh.cpp:30-49 */
    double *mn = b->nmin + 3 * (size_t)node, *mx = b->nmax + 3 * (size_t)node;
    for (int a = 0; a < 3; a++) { mn[a] = (double)1e30f; mx[a] = (double)-1e30f; }
    uint32_t first = b->first[node];
    for (uint32_t i = 0; i < b->count[node]; i++) {
        const double *t = b->tri + 9 * (size_t)b->index[first + i];
        for (int p = 0; p < 3; p++)
            for (int a = 0; a < 3; a++) mn[a] = MACRO_MIN(mn[a], t[3 * p + a]);
        for (int p = 0; p < 3; p++)
            for (int a = 0; a < 3; a++) mx[a] = MACRO_MAX(mx[a], t[3 * p + a]);
    }
}

static void subdivide(builder *b, uint32_t node) {                                       /* bvh.cpp:51-106 */
    if (b->count[node] <= 2) return;
    double ext[3];
    for (int a = 0; a < 3; a++) ext[a] = b->nmax[3 * (size_t)node + a] - b->nmin[3 * (size_t)node + a];
    int axis = 0;
    if (ext[1] > ext[0]) axis = 1;
    if (ext[2] > by_axis_f(ext, axis)) axis = 2;            /* double vs float-rounded compare :64 */
    float split = by_axis_f(b->nmin + 3 * (size_t)node, axis) + by_axis_f(ext, axis) * 0.5f;   /* :67 */
    int i = (int)b->first[node];
    int j = i + (int)b->count[node] - 1;
    while (i <= j) {
        if (by_axis_f(b->centroid + 3 * (size_t)b->index[i], axis) < split) {
            i++;
        } else {
            uint32_t t = b->index[i];
            b->index[i] = b->index[j];
            b->index[j--] = t;
        }
    }
    uint32_t left_count = (uint32_t)i - b->first[node];
    if (left_count == 0 || left_count == b->count[node]) return;
    uint32_t l = b->used++, r = b->used++;
    b->left[node] = l;
    b->first[l] = b->first[node];
    b->count[l] = left_count;
    b->first[r] = (uint32_t)i;
    b->count[r] = b->count[node] - left_count;
    b->count[node] = 0;
    update_bounds(b, l);
    update_bounds(b, r);
    subdivide(b, l);
    subdivide(b, r);
}

uint32_t ct_oracle_build_bvh(uint32_t n_tri, const double *tri, double *node_min, double *node_max,
                             uint32_t *node_left, uint32_t *node_first, uint32_t *node_count, uint32_t *tri_index) {
    builder b;
    b.n_tri = n_tri; b.tri = tri; b.used = 1;
    b.nmin = node_min; b.nmax = node_max; b.left = node_left; b.first = node_first; b.count = node_count; b.index = tri_index;
    size_t n_nodes = n_tri ? 2 * (size_t)n_tri - 1 : 1;
    memset(node_min, 0, n_nodes * 3 * sizeof(double));
    memset(node_max, 0, n_nodes * 3 * sizeof(double));
    memset(node_left, 0, n_nodes * sizeof(uint32_t));
    memset(node_first, 0, n_nodes * sizeof(uint32_t));
    memset(node_count, 0, n_nodes * sizeof(uint32_t));
    b.centroid = (double *)malloc(sizeof(double) * 3 * (size_t)(n_tri ? n_tri : 1));
    double third = (double)0.3333f;                         /* :112  (p1+p2+p3) * 0.3333f */
    for (uint32_t k = 0; k < n_tri; k++) {
        tri_index[k] = k;                                   /* :24-26 */
        const double *t = tri + 9 * (size_t)k;
        for (int a = 0; a < 3; a++) b.centroid[3 * (size_t)k + a] = third * ((t[a] + t[3 + a]) + t[6 + a]);
    }
    node_left[0] = 0; node_first[0] = 0; node_count[0] = n_tri;
    update_bounds(&b, 0);
    subdivide(&b, 0);
    free(b.centroid);
    return b.used;
}

/* ---- prototype (DESIGN.md, "what comes next" 1): the pre-hit phase of a closest-hit walk is order-free ----------
 * Until the first triangle test that changes ray.t (barycentric pass with 1e-4 < t < 1e30) the set of accepted boxes
 * is fixed, so WHICH triangle that is -- the one with the lowest leaf position among all such triangles reachable
 * through boxes accepted with ray.t = 1e30 -- can be found in any order.  From there the reference's walk is
 * reproduced by rebuilding its stack: the accepted right siblings along the root path of that leaf, deepest on top.
 * ct_oracle_closest_prehit does exactly that (phase 1 deliberately right-child-first) and must return what
 * ct_oracle_closest returns; tests/test_prehit_prototype.py checks it on every primary ray of the golden scenes. */
static void prehit_search(const ct_oracle_scene *s, const ray *r0, uint32_t node, uint32_t *best_pos) {
    if (!intersect_aabb(r0, s->node_min + 3 * (size_t)node, s->node_max + 3 * (size_t)node)) return;
    uint32_t count = s->node_count[node];
    if (count > 0) {
        uint32_t first = s->node_first[node];
        for (uint32_t i = 0; i < count && first + i < *best_pos; i++) {
            ray tmp = *r0;
            if (intersect_triangle(&tmp, s->tri + 9 * (size_t)s->tri_index[first + i]) && tmp.t != RAY_T_INIT) *best_pos = first + i;
        }
    } else {
        prehit_search(s, r0, s->node_left[node] + 1, best_pos);      /* any order will do: right child first */
        prehit_search(s, r0, s->node_left[node], best_pos);
    }
}

void ct_oracle_prehit_tables(const ct_oracle_scene *s, uint32_t *node_parent, uint32_t *leaf_of_pos) {
    node_parent[0] = 0xffffffffu;
    for (uint32_t n = 0; n < s->n_nodes; n++) {
        if (s->node_count[n] == 0) {
            if (s->node_left[n] + 1 < s->n_nodes) { node_parent[s->node_left[n]] = n; node_parent[s->node_left[n] + 1] = n; }
        } else {
            for (uint32_t i = 0; i < s->node_count[n]; i++) leaf_of_pos[s->node_first[n] + i] = n;
        }
    }
}

int ct_oracle_closest_prehit(const ct_oracle_scene *s, const uint32_t *node_parent, const uint32_t *leaf_of_pos,
                             const double org[3], const double dir[3], uint32_t *index, float *tclosest) {
    ctx cx; memset(&cx, 0, sizeof cx); cx.s = s;
    ray r = {v_load(org), v_load(dir), RAY_T_INIT};
    *tclosest = FINF;
    *index = 0;
    uint32_t best = 0xffffffffu;
    prehit_search(s, &r, 0, &best);
    if (best == 0xffffffffu) return 0;                              /* ray.t never changes: "not found" */
    /* the leaf of the first effective hit, tested as the reference tests it (the triangles before the hit change nothing) */
    uint32_t leaf = leaf_of_pos[best];
    for (uint32_t i = 0; i < s->node_count[leaf]; i++) {
        uint32_t k = s->tri_index[s->node_first[leaf] + i];
        int hit = intersect_triangle(&r, s->tri + 9 * (size_t)k);
        if (hit && r.t != RAY_T_INIT && r.t < *tclosest) { *index = k; *tclosest = r.t; }
    }
    /* the reference's pending work at that moment: right siblings of the left turns on the root path, accepted when
     * they were pushed (ray.t was still 1e30); the deepest is visited first, each re-tested against the current ray.t */
    ray r0 = {r.org, r.dir, RAY_T_INIT};
    for (uint32_t child = leaf, parent = node_parent[leaf]; parent != 0xffffffffu; child = parent, parent = node_parent[parent]) {
        if (child != s->node_left[parent]) continue;                 /* came from the right child: nothing pending here */
        uint32_t sib = child + 1;
        if (!intersect_aabb(&r0, s->node_min + 3 * (size_t)sib, s->node_max + 3 * (size_t)sib)) continue;
        bvh_closest(&cx, &r, sib, tclosest, index);
    }
    return r.t != RAY_T_INIT;
}

/* Both walks over n rays (ray.t = 1e30); returns the number of rays on which found / index / tclosest differ. */
uint64_t ct_oracle_prehit_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, uint64_t *n_found) {
    uint32_t *node_parent = (uint32_t *)malloc((size_t)s->n_nodes * sizeof(uint32_t));
    uint32_t *leaf_of_pos = (uint32_t *)malloc((size_t)s->n_tri * sizeof(uint32_t));
    ct_oracle_prehit_tables(s, node_parent, leaf_of_pos);
    uint64_t bad = 0, found = 0;
    for (uint64_t i = 0; i < n; i++) {
        uint32_t ia, ib; float ta, tb;
        int fa = ct_oracle_closest(s, org + 3 * i, dir + 3 * i, RAY_T_INIT, &ia, &ta);
        int fb = ct_oracle_closest_prehit(s, node_parent, leaf_of_pos, org + 3 * i, dir + 3 * i, &ib, &tb);
        found += (uint64_t)fa;
        if (fa != fb || ia != ib || memcmp(&ta, &tb, sizeof ta) != 0) bad++;
    }
    free(node_parent); free(leaf_of_pos);
    if (n_found) *n_found = found;
    return bad;
}

/* ---- prototype: the WHOLE closest-hit walk as an order-free search + a replay of the near-minimum candidates ----------
 * (what cobbletrace_b200's k_primary_split does on the device; checked here, on the CPU, against bvh_closest.)
 * On a nested tree the reference tests triangle Z iff its LEAF's box passes IntersectAABB against the ray.t of that moment
 * (DESIGN.md 2).  With G = the triangles with a barycentric pass and 1e-4 < t < 1e30 in leaves whose box passes the two
 * conditions that do not depend on ray.t, and m = min t over G:
 *   * ray.t never drops below m, and ends at <= m + sigma, where sigma bounds  tmin(leaf box of Z) - t_Z  over all Z
 *     (a triangle lies inside its leaf's box, so only rounding can make its t smaller than the box's entry distance);
 *   * a triangle with t > tau can change the fate of one with t <= tau only by blocking its leaf, i.e. only if that
 *     leaf's tmin >= t > tau.
 * So: find, in ANY order and pruning boxes whose tmin > best + 2 sigma, every member of G with t <= m + sigma (= S); if
 * every member of S has tmin(leaf) <= m + sigma, replaying the reference's update rules over S alone, in leaf-position
 * order, yields the reference's ray.t / tclosest / closestIndex.  Otherwise (and for m >= FINF) the caller falls back to
 * the ordered walk.  order: 0 = left child first, 1 = nearer child first.
 * stats[0] += box tests, stats[1] += triangle tests, stats[2] += fallbacks, stats[3] = max |S| seen. */
typedef struct { float t, tmin; uint32_t pos, leaf; } free_cand;
typedef struct {
    const ct_oracle_scene *s; const ray *r; double sigma; double best;
    free_cand cand[64]; int n_cand, overflow; uint64_t *stats;
} free_ctx;

static int box_times_ref(const ray *r, const double *bmin, const double *bmax, float *tmin_out) {
    float tx1 = (float)((bmin[0] - r->org.x) / r->dir.x), tx2 = (float)((bmax[0] - r->org.x) / r->dir.x);
    float tmin = MACRO_MIN(tx1, tx2), tmax = MACRO_MAX(tx1, tx2);
    float ty1 = (float)((bmin[1] - r->org.y) / r->dir.y), ty2 = (float)((bmax[1] - r->org.y) / r->dir.y);
    tmin = MACRO_MAX(tmin, MACRO_MIN(ty1, ty2)); tmax = MACRO_MIN(tmax, MACRO_MAX(ty1, ty2));
    float tz1 = (float)((bmin[2] - r->org.z) / r->dir.z), tz2 = (float)((bmax[2] - r->org.z) / r->dir.z);
    tmin = MACRO_MAX(tmin, MACRO_MIN(tz1, tz2)); tmax = MACRO_MIN(tmax, MACRO_MAX(tz1, tz2));
    *tmin_out = tmin;
    return tmax >= tmin && tmax > 0;
}

static void free_leaf(free_ctx *c, uint32_t node, float leaf_tmin) {
    const ct_oracle_scene *s = c->s;
    uint32_t first = s->node_first[node];
    for (uint32_t i = 0; i < s->node_count[node]; i++) {
        ray tmp = *c->r; tmp.t = RAY_T_INIT;
        c->stats[1]++;
        if (!intersect_triangle(&tmp, s->tri + 9 * (size_t)s->tri_index[first + i]) || tmp.t == RAY_T_INIT) continue;
        if ((double)tmp.t > c->best + c->sigma) continue;
        if ((double)tmp.t < c->best) c->best = (double)tmp.t;
        if (c->n_cand == 64) {                                   /* drop what has fallen out of the band */
            int k = 0;
            for (int j = 0; j < c->n_cand; j++) if ((double)c->cand[j].t <= c->best + c->sigma) c->cand[k++] = c->cand[j];
            c->n_cand = k;
            if (k == 64) { c->overflow = 1; continue; }
        }
        free_cand z = {tmp.t, leaf_tmin, first + i, node};
        c->cand[c->n_cand++] = z;
    }
}

static void free_walk(free_ctx *c, uint32_t node, float node_tmin, int order) {
    const ct_oracle_scene *s = c->s;
    if ((double)node_tmin > c->best + 2.0 * c->sigma) return;                     /* the deferred distance test */
    if (s->node_count[node] > 0) { free_leaf(c, node, node_tmin); return; }
    uint32_t l = s->node_left[node], rgt = l + 1;
    float tl, tr;
    c->stats[0] += 2;
    int hl = box_times_ref(c->r, s->node_min + 3 * (size_t)l, s->node_max + 3 * (size_t)l, &tl);
    int hr = box_times_ref(c->r, s->node_min + 3 * (size_t)rgt, s->node_max + 3 * (size_t)rgt, &tr);
    if (order == 1 && hl && hr && tr < tl) {
        free_walk(c, rgt, tr, order); free_walk(c, l, tl, order);
    } else {
        if (hl) free_walk(c, l, tl, order);
        if (hr) free_walk(c, rgt, tr, order);
    }
}

/* Returns found (0 / 1), or -1 when the ordered walk must decide (*index / *tclosest untouched then). */
int ct_oracle_closest_free(const ct_oracle_scene *s, const double org[3], const double dir[3], int order,
                           uint32_t *index, float *tclosest, uint64_t *stats) {
    ray r = {v_load(org), v_load(dir), RAY_T_INIT};
    free_ctx c; memset(&c, 0, sizeof c);
    c.s = s; c.r = &r; c.stats = stats; c.best = (double)RAY_T_INIT;
    double m = 0;
    for (int a = 0; a < 3; a++) {
        double bound = 0;
        bound = fmax(fabs(s->node_min[a]), fabs(s->node_max[a]));                  /* node 0 holds every triangle */
        double mk = (bound + fabs(org[a])) / fabs(dir[a]);
        if (!(mk < 1e30)) { stats[2]++; return -1; }                               /* zero / non-finite direction component */
        m = fmax(m, mk);
    }
    c.sigma = m * 0x1p-15;                                 /* as tray_nearest_setup (ct_exact.cuh) */
    float t0;
    stats[0]++;
    if (!box_times_ref(&r, s->node_min, s->node_max, &t0)) { *index = 0; *tclosest = FINF; return 0; }
    free_walk(&c, 0, t0, order);
    if (c.overflow) { stats[2]++; return -1; }
    if (c.best == (double)RAY_T_INIT) { *index = 0; *tclosest = FINF; return 0; }
    if (c.best >= (double)FINF) { stats[2]++; return -1; }
    const double tau = c.best + c.sigma;
    int n = 0;
    for (int j = 0; j < c.n_cand; j++) if ((double)c.cand[j].t <= tau) c.cand[n++] = c.cand[j];
    if ((uint64_t)n > stats[3]) stats[3] = (uint64_t)n;
    for (int j = 0; j < n; j++) if (!((double)c.cand[j].tmin <= tau)) { stats[2]++; return -1; }
    for (int j = 1; j < n; j++) {                                                  /* leaf-position order = the reference's test order */
        free_cand z = c.cand[j]; int k = j;
        while (k > 0 && c.cand[k - 1].pos > z.pos) { c.cand[k] = c.cand[k - 1]; k--; }
        c.cand[k] = z;
    }
    float rt = RAY_T_INIT, tc = FINF; uint32_t idx = 0;
    uint32_t entered = 0xffffffffu;                                                /* the box is tested once per leaf visit, not per triangle */
    for (int j = 0; j < n; j++) {
        if (c.cand[j].leaf != entered) {
            if (!(c.cand[j].tmin < rt)) continue;                                  /* bvh.cpp:178 for the leaf's own box */
            entered = c.cand[j].leaf;
        }
        rt = MACRO_MIN(rt, c.cand[j].t);                                           /* bvh.cpp:161 (t > 1e-4 by construction) */
        if (rt != RAY_T_INIT && rt < tc) { idx = s->tri_index[c.cand[j].pos]; tc = rt; }   /* bvh.cpp:212 */
    }
    *index = idx; *tclosest = tc;
    return rt != RAY_T_INIT;
}

/* Both walks over n rays; returns how many rays the free walk answered differently (fallbacks excluded, counted in stats[2]).
 * ref_stats[0] / [1] += the reference walk's box / triangle tests. */
uint64_t ct_oracle_free_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, int order,
                              uint64_t *stats, uint64_t *ref_stats) {
    uint64_t bad = 0;
    for (uint64_t i = 0; i < n; i++) {
        uint32_t ia = 0, ib = 0; float ta = 0, tb = 0;
        ctx cx; memset(&cx, 0, sizeof cx); cx.s = s;
        ray r = {v_load(org + 3 * i), v_load(dir + 3 * i), RAY_T_INIT};
        ta = FINF; ia = 0;
        bvh_closest(&cx, &r, 0, &ta, &ia);
        int fa = r.t != RAY_T_INIT;
        ref_stats[0] += cx.c.box_tests; ref_stats[1] += cx.c.tri_tests;
        int fb = ct_oracle_closest_free(s, org + 3 * i, dir + 3 * i, order, &ib, &tb, stats);
        if (fb < 0) continue;
        if (fa != fb || ia != ib || memcmp(&ta, &tb, sizeof ta) != 0) bad++;
    }
    return bad;
}

/* ---- prototype: ONE long closest-hit walk split across the 32 lanes of a warp (DESIGN.md 8, "long walks split across a warp") --------
 * The order-free formulation above lets a walk be processed as a frontier: per ROUND up to 32 pending nodes are taken off a shared
 * stack (one per lane), their children tested against best + 2 sigma, accepted leaves tested on the spot (candidates as above),
 * accepted interior children pushed back; the warp-wide minimum of t is taken once per round.  A round costs about what one visit of
 * the ordered walk costs (~1 us on the device), so `rounds` against the ordered walk's pair visits is the floor such a kernel would
 * have against today's.  Returns found / -1 like ct_oracle_closest_free; *rounds and *pair_visits are set either way. */
int ct_oracle_closest_rounds(const ct_oracle_scene *s, const double org[3], const double dir[3], uint32_t *index, float *tclosest,
                             uint32_t *rounds, uint32_t *pair_visits) {
    ray r = {v_load(org), v_load(dir), RAY_T_INIT};
    uint64_t stats[4] = {0, 0, 0, 0};
    free_ctx c; memset(&c, 0, sizeof c);
    c.s = s; c.r = &r; c.stats = stats; c.best = (double)RAY_T_INIT;
    *rounds = 0; *pair_visits = 0;
    double m = 0;
    for (int a = 0; a < 3; a++) {
        double bound = fmax(fabs(s->node_min[a]), fabs(s->node_max[a]));
        double mk = (bound + fabs(org[a])) / fabs(dir[a]);
        if (!(mk < 1e30)) return -1;
        m = fmax(m, mk);
    }
    c.sigma = m * 0x1p-15;                                 /* as tray_nearest_setup (ct_exact.cuh) */
    float t0;
    if (!box_times_ref(&r, s->node_min, s->node_max, &t0)) { *index = 0; *tclosest = FINF; return 0; }
    enum { CAP = 4096 };
    static __thread uint32_t stk[CAP];
    static __thread float stk_t[CAP];
    uint32_t sp = 0;
    if (s->node_count[0] > 0) free_leaf(&c, 0, t0); else { stk[sp] = 0; stk_t[sp] = t0; sp++; }
    while (sp > 0) {
        uint32_t take = sp < 32 ? sp : 32;
        sp -= take;
        uint32_t out[64]; float out_t[64]; uint32_t n_out = 0;
        const double thr = c.best + 2.0 * c.sigma;                      /* the warp-wide minimum: once per round */
        double best_round = c.best;
        (*rounds)++;
        for (uint32_t l = 0; l < take; l++) {                           /* "lanes" */
            uint32_t node = stk[sp + l];
            if ((double)stk_t[sp + l] > thr) continue;
            (*pair_visits)++;
            for (uint32_t ch = s->node_left[node]; ch <= s->node_left[node] + 1; ch++) {
                float tc;
                if (!box_times_ref(&r, s->node_min + 3 * (size_t)ch, s->node_max + 3 * (size_t)ch, &tc)) continue;
                if ((double)tc > thr) continue;
                if (s->node_count[ch] > 0) {
                    double keep = c.best;                               /* lanes see each other's hits at the round's end only */
                    c.best = best_round;
                    free_leaf(&c, ch, tc);
                    if (c.best < keep) keep = c.best;
                    best_round = c.best < best_round ? c.best : best_round;
                    c.best = keep < best_round ? keep : best_round;
                } else { out[n_out] = ch; out_t[n_out] = tc; n_out++; }
            }
        }
        if (sp + n_out > CAP) return -1;
        for (uint32_t k = 0; k < n_out; k++) { stk[sp] = out[k]; stk_t[sp] = out_t[k]; sp++; }
    }
    if (c.overflow) return -1;
    if (c.best == (double)RAY_T_INIT) { *index = 0; *tclosest = FINF; return 0; }
    if (c.best >= (double)FINF) return -1;
    const double tau = c.best + c.sigma;
    int n = 0;
    for (int j = 0; j < c.n_cand; j++) if ((double)c.cand[j].t <= tau) c.cand[n++] = c.cand[j];
    for (int j = 0; j < n; j++) if (!((double)c.cand[j].tmin <= tau)) return -1;
    for (int j = 1; j < n; j++) {
        free_cand z = c.cand[j]; int k = j;
        while (k > 0 && c.cand[k - 1].pos > z.pos) { c.cand[k] = c.cand[k - 1]; k--; }
        c.cand[k] = z;
    }
    float rt = RAY_T_INIT, tc = FINF; uint32_t idx = 0, entered = 0xffffffffu;
    for (int j = 0; j < n; j++) {
        if (c.cand[j].leaf != entered) {
            if (!(c.cand[j].tmin < rt)) continue;
            entered = c.cand[j].leaf;
        }
        rt = MACRO_MIN(rt, c.cand[j].t);
        if (rt != RAY_T_INIT && rt < tc) { idx = s->tri_index[c.cand[j].pos]; tc = rt; }
    }
    *index = idx; *tclosest = tc;
    return rt != RAY_T_INIT;
}

/* Over n rays: the ordered walk's pair visits (= box tests / 2) against the frontier walk's rounds, for the rays whose ordered walk
 * needs at least min_visits pair visits.  out[0] rays considered, out[1] differing answers (must be 0), out[2] undecided, out[3] sum of
 * ordered pair visits, out[4] sum of rounds, out[5] max ordered pair visits, out[6] max rounds, out[7] rounds of the longest ordered walk. */
void ct_oracle_rounds_check(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, uint32_t min_visits, uint64_t out[8]) {
    memset(out, 0, 8 * sizeof(uint64_t));
    for (uint64_t i = 0; i < n; i++) {
        ctx cx; memset(&cx, 0, sizeof cx); cx.s = s;
        ray r = {v_load(org + 3 * i), v_load(dir + 3 * i), RAY_T_INIT};
        float ta = FINF; uint32_t ia = 0;
        bvh_closest(&cx, &r, 0, &ta, &ia);
        int fa = r.t != RAY_T_INIT;
        uint64_t visits = cx.c.box_tests / 2;
        if (visits < min_visits) continue;
        uint32_t ib = 0, rounds = 0, pv = 0; float tb = 0;
        int fb = ct_oracle_closest_rounds(s, org + 3 * i, dir + 3 * i, &ib, &tb, &rounds, &pv);
        out[0]++;
        if (fb < 0) { out[2]++; continue; }
        if (fa != fb || ia != ib || memcmp(&ta, &tb, sizeof ta) != 0) out[1]++;
        out[3] += visits; out[4] += rounds;
        if (visits > out[5]) { out[5] = visits; out[7] = rounds; }
        if (rounds > out[6]) out[6] = rounds;
    }
}

/* ---- the slop bound of the order-free walk, measured: for n (ray, triangle) cases the box of the triangle alone (the tightest leaf box the
 * builder can produce, bvh.cpp:30-49) against the triangle's own t, both in the reference's arithmetic.  out[0] = barycentric passes with
 * 1e-4 < t < 1e30, out[1] = max over them of (tmin(box) - t) / M with M = max_k (bound_k + |o_k|) / |d_k| as tray_nearest_setup defines it
 * (bound_k = the largest |coordinate| of the triangle on axis k), out[2] = cases skipped for being outside the analysis' magnitude limits. */
void ct_oracle_slop_check(uint64_t n, const double *org, const double *dir, const double *tri, double out[3]) {
    out[0] = out[1] = out[2] = 0;
    double worst = -1e300;
    for (uint64_t i = 0; i < n; i++) {
        const double *o = org + 3 * i, *d = dir + 3 * i, *t = tri + 9 * i;
        double bmin[3], bmax[3], bound[3], M = 0, B = 0, O = 0, D = 0;
        int ok = 1;
        for (int a = 0; a < 3; a++) {
            bmin[a] = fmin(fmin(t[a], t[3 + a]), t[6 + a]); bmax[a] = fmax(fmax(t[a], t[3 + a]), t[6 + a]);
            bound[a] = fmax(fabs(bmin[a]), fabs(bmax[a]));
            if (!(fabs(d[a]) > 0)) ok = 0;
            M = fmax(M, (bound[a] + fabs(o[a])) / fabs(d[a]));
            B = fmax(B, bound[a]); O = fmax(O, fabs(o[a])); D = fmax(D, fabs(d[a]));
        }
        if (!ok || !(D * B * B <= 4096.0) || !((O + B) * D * B <= 4096.0) || !(M < 0x1p60)) { out[2]++; continue; }
        ray r = {v_load(o), v_load(d), RAY_T_INIT};
        if (!intersect_triangle(&r, t) || r.t == RAY_T_INIT) continue;
        float tmin;
        ray r0 = {v_load(o), v_load(d), RAY_T_INIT};
        box_times_ref(&r0, bmin, bmax, &tmin);
        out[0]++;
        double ratio = ((double)tmin - (double)r.t) / M;
        if (ratio > worst) worst = ratio;
    }
    out[1] = worst;
}
