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
