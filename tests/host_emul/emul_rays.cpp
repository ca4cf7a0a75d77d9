// TEST INFRASTRUCTURE ONLY -- the primary pass of a batch of caller-given rays (render_rays_kernel: trace_core.cuh's
// given_ray_color) on the host, compiled into tests/host_emul/libhostemul_rays.so (tests/emul_rays_lib.py).  It builds on
// emul.cpp (scene setup, the emitter, the dimension dispatch), which is included whole, and adds two entry points:
//   emul_rays_vs_plain  the camera's own rays through given_ray_color next to the plain primary pass: colour bits, bounce
//                       records and counters must be identical;
//   emul_render_rays    a whole rays call: the ray-fed primary pass, then one pass per reflection depth, with the AOVs.
#include "emul.cpp"

namespace {

template <int DT>
bool same_records(const std::vector<Bounce<DT>> &a, const std::vector<Bounce<DT>> &b, int D) {
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i) {
        if (memcmp(a[i].o, b[i].o, sizeof(float) * D) || memcmp(a[i].d, b[i].d, sizeof(float) * D) ||
            memcmp(a[i].w, b[i].w, sizeof a[i].w) || a[i].skip.ref != b[i].skip.ref || a[i].skip.lane != b[i].skip.lane ||
            a[i].depth != b[i].depth)
            return false;
    }
    return true;
}

void put_counters(unsigned long long *o, const Counters &c) {
    o[0] = c.reflection_rays; o[1] = c.shadow_rays; o[2] = c.node_steps; o[3] = c.simplex_tests;
    o[4] = c.solid_tests; o[5] = c.shaded_hits; o[6] = c.truncated;
}

template <int DT, int FLAGS>
void vs_plain_t(Scene &S, int w, int h, float *rgb_plain, float *rgb_rays, float *rays_out, unsigned long long *cnt,
                unsigned long long *rec) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = S.dev.dim;
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = 1;
    f.width = w; f.height = h;
    f.half_w = (float)w / 2.0f; f.half_h = (float)h / 2.0f;
    f.fovI = tanf(S.dev.fov / 2) / f.half_w;
    Counters c1, c2;
    std::vector<Bounce<DT>> q1, q2;
    std::vector<uint32_t> p1, p2;
    const float one[3] = {1, 1, 1};
    const Skip none = {NTR_NONE_REF, 0};
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            const uint32_t pix = (uint32_t)y * w + x;
            // the plain builds (kernels.cuh, render_pass_kernel without NTR_F_SS / NTR_F_VIEWS)
            float o[CAP], dir[CAP], acc[3] = {0, 0, 0};
            HitRec prim;
            prim.dist = 0; prim.ref = NTR_NONE_REF; prim.lane = -1;
            primary_ray_of<DT>(S.dev, S.cam, f.fovI, f.half_w, f.half_h, x, y, o, dir);
            if (S.dev.kind == NTR_SCENE_BOX) box_color<DT>(S.dev, o, dir, acc, &prim);
            else {
                VecEmit<DT> emit{&q1, &p1, pix};
                ray_color<DT, FLAGS>(S.dev, true, o, dir, 0, none, one, acc, emit, c1, &prim, &ms);
            }
            rgb_plain[pix * 3] = acc[0]; rgb_plain[pix * 3 + 1] = acc[1]; rgb_plain[pix * 3 + 2] = acc[2];
            // the same ray handed in from memory (render_rays_kernel)
            memcpy(rays_out + (size_t)pix * 2 * D, o, sizeof(float) * D);
            memcpy(rays_out + (size_t)pix * 2 * D + D, dir, sizeof(float) * D);
            float ro[CAP], rd[CAP];
            for (int k = 0; k < D; ++k) { ro[k] = rays_out[(size_t)pix * 2 * D + k]; rd[k] = rays_out[(size_t)pix * 2 * D + D + k]; }
            VecEmit<DT> emit{&q2, &p2, pix};
            given_ray_color<DT, FLAGS>(S.dev, ro, rd, rgb_rays + (size_t)pix * 3, emit, c2, &ms, (PrimaryAov<DT> *)nullptr);
        }
    }
    ms.detach();
    put_counters(cnt, c1);
    put_counters(cnt + 7, c2);
    rec[0] = q1.size(); rec[1] = q2.size();
    rec[2] = same_records<DT>(q1, q2, D) && p1 == p2;
}

template <int DT, int FLAGS>
void rays_t(Scene &S, uint32_t n, const float *origins, const float *dirs, float *rgb, int32_t *ids, float *dist,
            float *normals, unsigned long long *cnt) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = S.dev.dim;
    Counters c;
    std::vector<Bounce<DT>> q, qn;
    std::vector<uint32_t> qp, qpn;
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    for (uint32_t i = 0; i < n; ++i) {
        float o[CAP], dir[CAP];
        for (int k = 0; k < D; ++k) { o[k] = origins[(size_t)i * D + k]; dir[k] = dirs[(size_t)i * D + k]; }
        VecEmit<DT> emit{&q, &qp, i};
        PrimaryAov<DT> a;
        given_ray_color<DT, FLAGS>(S.dev, o, dir, rgb + (size_t)i * 3, emit, c, &ms, &a);
        // store_aov (kernels.cuh)
        const bool hit = a.hit.ref != NTR_NONE_REF;
        ids[i] = !hit ? -1 : (S.dev.kind == NTR_SCENE_BOX ? 0 : flat_prim_id(S.dev, a.hit.ref, a.hit.lane));
        dist[i] = a.hit.dist;
        for (int k = 0; k < D; ++k) normals[(size_t)i * D + k] = a.n[k];
    }
    while (!q.empty()) {
        qn.clear(); qpn.clear();
        for (size_t i = 0; i < q.size(); ++i) {
            float acc[3] = {0, 0, 0};
            VecEmit<DT> emit{&qn, &qpn, qp[i]};
            ray_color<DT, FLAGS>(S.dev, true, q[i].o, q[i].d, q[i].depth, q[i].skip, q[i].w, acc, emit, c, nullptr, &ms);
            rgb[(size_t)qp[i] * 3] += acc[0]; rgb[(size_t)qp[i] * 3 + 1] += acc[1]; rgb[(size_t)qp[i] * 3 + 2] += acc[2];
        }
        q.swap(qn); qp.swap(qpn);
    }
    ms.detach();
    put_counters(cnt, c);
}

}  // namespace

extern "C" {

// A w x h frame's primary pass two ways: the plain pass, and the camera's rays (primary_ray_of, written to rays: w*h x 2 x D
// floats, origin then direction) through given_ray_color.  rgb_plain / rgb_rays: w*h*3 floats; counters: 2 x 7 words
// (reflection, shadow, node steps, simplex tests, solid tests, shaded hits, truncated), plain then rays; records: [0] plain
// count, [1] rays count, [2] 1 if identical (bounce records and their pixel words).
__attribute__((visibility("default"))) int emul_rays_vs_plain(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                               int w, int h, int force_generic, float *rgb_plain, float *rgb_rays,
                                                               float *rays, unsigned long long *counters, unsigned long long *records) {
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                            \
    if (S.flags & NTR_F_GENERAL) vs_plain_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, w, h, rgb_plain, rgb_rays, rays, counters, records); \
    else vs_plain_t<DT, NTR_F_COUNT>(S, w, h, rgb_plain, rgb_rays, rays, counters, records);
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

// A rays call of n rays (origins / dirs n x D): colours (n x 3) after every bounce pass, the AOVs (ids, dist: n; normals:
// n x D) and the counters (7 words as above).
__attribute__((visibility("default"))) int emul_render_rays(const ntr_scene_desc *d, uint32_t n, const float *origins, const float *dirs,
                                                             int force_generic, float *rgb, int32_t *ids, float *dist, float *normals,
                                                             unsigned long long *counters) {
    Scene S;
    setup(S, d, nullptr, nullptr);
#define CALL(DT)                                                                                                            \
    if (S.flags & NTR_F_GENERAL) rays_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, n, origins, dirs, rgb, ids, dist, normals, counters); \
    else rays_t<DT, NTR_F_COUNT>(S, n, origins, dirs, rgb, ids, dist, normals, counters);
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

}  // extern "C"
