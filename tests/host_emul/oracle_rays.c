/* TEST INFRASTRUCTURE ONLY -- the oracle's answer for a batch of caller-given primary rays (ntr_render_rays), compiled into
 * tests/host_emul/liboracle_rays.so (tests/oracle_rays_lib.py).  It includes the C restatement of the reference
 * (oracle/ntr_oracle.c) whole, so that it uses the oracle's own aabb_distance, ray_color and traversal, and adds one entry
 * point; the oracle itself is left as it is. */
#include "../../oracle/ntr_oracle.c"

/* The colour of n caller-given primary rays (ntr_render_rays): box_scene::calculate_color's colour of the ray, or
 * composite_scene::ray_color(ray, 0, none) (tracer.hpp:101-114, 1856-1883), and the opaque hit as the render path sees it,
 * intersects(root, ray, {}, ..., aabb_distance, max).  rgb: n x 3.  Optional: ids / dist (-1 / 0 on a miss), t0 (the ray's
 * aabb_distance, -1 where it misses the scene box; 0 for BoxScenes), undefined_mask (per ray, as oracle_render_float's),
 * counters (primary_rays = n). */
ORACLE_API int oracle_ray_colors(const ntr_scene_desc *s, uint32_t n, const float *origins, const float *dirs, float *rgb,
                                 int32_t *ids, float *dist, float *t0, uint8_t *undefined_mask, ntr_counters *counters) {
    ntr_counters total;
    memset(&total, 0, sizeof total);
#pragma omp parallel
    {
        octx c;
        ctx_init(&c, s, NULL, NULL);
#pragma omp for schedule(dynamic, 16)
        for (uint32_t i = 0; i < n; ++i) {
            const int D = c.D;
            oray view;
            memcpy(view.o, origins + (size_t)i * D, sizeof(float) * D);
            memcpy(view.d, dirs + (size_t)i * D, sizeof(float) * D);
            c.undefined = 0;
            c.cnt.primary_rays++;
            ocolor r;
            int32_t id = -1;
            float hd = 0, t = 0;
            if (s->kind == NTR_SCENE_BOX) {
                oray normal;
                memset(&normal, 0, sizeof normal);
                float d = hypercube_intersects(D, &view, &normal, FLT_MAX);
                if (d) {
                    float sine = dotD(D, view.d, normal.d);
                    r = cmulf(col(1, 0.5f, 0.5f), sine <= 0 ? -sine : 0.0f);
                    id = 0;
                    hd = d;
                } else {
                    float intensity = view.d[0];
                    r = intensity > 0 ? col(intensity, intensity, intensity) : col(0, -intensity, -intensity);
                }
            } else {
                otarget none = { NONE_REF, 0 };
                ntr_counters keep = c.cnt;
                t = aabb_distance(&c, &view);
                if (t >= 0) {
                    ohit hit;
                    memset(&hit, 0, sizeof hit);
                    hit.dist = FLT_MAX;
                    ohits th = { NULL, 0, 0 };
                    if (tree_intersects(&c, s->root, &view, none, &hit, &th, t, FLT_MAX)) { id = flat_id(s, hit.target); hd = hit.dist; }
                    free(th.v);
                }
                c.cnt = keep;           /* the hit lookup is not part of the colour's work */
                r = ray_color(&c, &view, 0, none);
            }
            rgb[(size_t)i * 3] = r.r; rgb[(size_t)i * 3 + 1] = r.g; rgb[(size_t)i * 3 + 2] = r.b;
            if (ids) ids[i] = id;
            if (dist) dist[i] = hd;
            if (t0) t0[i] = t;
            if (undefined_mask) undefined_mask[i] = (uint8_t)c.undefined;
        }
#pragma omp critical
        cnt_add(&total, &c.cnt);
    }
    if (counters) *counters = total;
    return 0;
}
