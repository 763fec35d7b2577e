/* lens_oracle.c -- TEST INFRASTRUCTURE: the oracle's Scene::Render (oracle/rt_oracle.c orc_render_sum) with the thin
 * lens of rtc_scene_set_lens in its camera sample, restated in C for tests/test_lens.py.  The oracle itself restates the
 * reference, which has no lens, and stays as it is; this file compiles it in and adds the lens step.
 *
 * The lens step (DESIGN.md "Thin lens"): b = the slot-0 Philox block of (pixel, sample), whose b[0], b[1] give the
 * jitter; (lx, ly) = concentric map of u01(b[2]), u01(b[3]); e = lx right + ly up; origin pos + r e, direction
 * d - (r / f) e.  sin / cos of the map are evaluated in double here and by sincospif (1 ulp) on the device: the lens point
 * may differ by an ulp, so a ray may differ in its last bits and, rarely, a path may take another branch. */
#include "../../oracle/rt_oracle.c"

static void lens_disk(float u, float v, float* lx, float* ly) {
    const float sx = 2.f * u - 1.f, sy = 2.f * v - 1.f;
    if (sx == 0.f && sy == 0.f) { *lx = 0.f; *ly = 0.f; return; }
    float rad, th;
    if (fabsf(sx) > fabsf(sy)) { rad = sx; th = 0.25f * (sy / sx); }
    else { rad = sy; th = 0.5f - 0.25f * (sx / sy); }
    *lx = rad * (float)cos(3.141592653589793 * (double)th);
    *ly = rad * (float)sin(3.141592653589793 * (double)th);
}

/* orc_render_sum with a lens of aperture radius r focused at f (r = 0: orc_render_sum's sums bit for bit) */
void orc_render_sum_lens(const orc_scene* s, float r, float f, uint32_t seed, uint32_t sample_begin, uint32_t sample_count,
                         long pix_begin, long pix_end, float* out_sum, uint64_t counters[2], int nthreads) {
    uint64_t paths = 0, rays = 0;
    const float k = r / f;
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#else
    (void)nthreads;
#endif
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : paths, rays)
    for (long i = pix_begin; i < pix_end; ++i) {
        unsigned x = (unsigned)(i % s->width), y = (unsigned)(i / s->width);
        v3 sum = V(0, 0, 0);
        for (uint32_t j = 0; j < sample_count; ++j) {
            uint32_t smp = sample_begin + j;
            rng_t g = {seed, (uint32_t)i, smp, 0};
            uint32_t b[4]; rng_block(&g, 0, b);
            float fx = (float)x + u01(b[0]), fy = (float)y + u01(b[1]);
            if (s->dialect == 3) { fx = (float)((double)fx + 0.5); fy = (float)((double)fy + 0.5); }
            ray_t ray = cam_ray(s, fx, fy);
            if (r > 0.f) {
                float lx, ly;
                lens_disk(u01(b[2]), u01(b[3]), &lx, &ly);
                const v3 e = vadd(vscale(lx, s->cam_right), vscale(ly, s->cam_up));
                ray.o = vadd(ray.o, vscale(r, e));
                ray.d = V(ray.d.x - k * e.x, ray.d.y - k * e.y, ray.d.z - k * e.z);
            }
            uint64_t nr = 0;
            v3 c = ray_trace(s, seed, (uint32_t)i, smp, ray, &nr);
            sum = vadd(sum, c);
            paths++; rays += nr;
        }
        out_sum[3 * (i - pix_begin) + 0] = sum.x;
        out_sum[3 * (i - pix_begin) + 1] = sum.y;
        out_sum[3 * (i - pix_begin) + 2] = sum.z;
    }
    if (counters) { counters[0] += paths; counters[1] += rays; }
}
