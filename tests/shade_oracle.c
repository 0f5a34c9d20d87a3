/* tests/shade_oracle.c -- ct_oracle_trace_many: the oracle's TraceRay (raythread.cpp:353-386) for caller rays, the checker of
 * tests/test_shade_rays.py.  It compiles the pinned restatement oracle/ct_oracle.c as it stands (included, not copied) and only
 * exposes its `static trace_ray`, so the colours come from exactly the code tests/test_oracle_golden.py pins to the reference.
 * Build: cc -O2 -ffp-contract=off -fno-fast-math -fPIC -shared -std=c11 -I oracle tests/shade_oracle.c -lm -lpthread
 * (the flags of oracle/Makefile's restatement). */
#include "ct_oracle.c"

/* color[i] = TraceRay({org[i], dir[i], ray.t = 1e30f}, 1, FINF, max_depth), 0x00BBGGRR: what a primary ray of a frame gets
 * (trace_canvas_point), for any origin and direction. */
void ct_oracle_trace_many(const ct_oracle_scene *s, uint64_t n, const double *org, const double *dir, int max_depth, uint32_t *color) {
    for (uint64_t i = 0; i < n; i++) {
        ctx cx;
        memset(&cx, 0, sizeof cx);
        cx.s = s;
        ray r = {v_load(org + 3 * i), v_load(dir + 3 * i), RAY_T_INIT};
        color[i] = trace_ray(&cx, r, max_depth);
    }
}

/* ---- the shading arithmetic case by case: the checkers of tests/test_shading_kat.py ------------------------------------------------ */
void ct_oracle_shade_many(uint64_t n, const uint32_t *color, const float *intensity, uint32_t *out) {
    for (uint64_t i = 0; i < n; i++) out[i] = ct_oracle_shade_color(color[i], intensity[i]);
}

void ct_oracle_blend_many(uint64_t n, const uint32_t *lc, const uint32_t *rc, const float *reflection, uint32_t *out) {
    for (uint64_t i = 0; i < n; i++) out[i] = ct_oracle_blend(lc[i], rc[i], reflection[i]);
}

/* pw[i] = glibc's pow(x, e) as compute_lighting calls it; acc_out[i] (when acc_out is not NULL) = its accumulation of the term. */
void ct_oracle_pow_many(uint64_t n, const float *x, const int32_t *e, const float *acc, const float *li, double *pw, float *acc_out) {
    for (uint64_t i = 0; i < n; i++) {
        double p = pow((double)x[i], (double)e[i]);
        pw[i] = p;
        if (acc_out) acc_out[i] = (float)((double)acc[i] + (double)li[i] * p);
    }
}

/* The conversion the oracle writes, (uint8_t)(int)c, next to a direct double -> uint8_t assignment, both compiled with the flags above. */
void ct_oracle_u8_forms(uint64_t n, const double *c, uint8_t *via_int, uint8_t *direct) {
    for (uint64_t i = 0; i < n; i++) {
        via_int[i] = (uint8_t)(int)c[i];
        direct[i] = c[i];
    }
}
