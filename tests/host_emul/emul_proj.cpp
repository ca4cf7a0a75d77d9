// TEST INFRASTRUCTURE ONLY -- projected frames (ntr_scene_set_projection) on the host, compiled into
// tests/host_emul/libhostemul_proj.so (tests/emul_proj_lib.py).  It builds on emul.cpp (scene setup, the emitter, the
// dimension dispatch), which is included whole, and adds three entry points:
//   emul_camera_rays     camera_rays_kernel: primary_ray with PROJ for every pixel of a view;
//   emul_render_proj     a whole projected frame at factor s, full or adaptive: the primary pass of the NTR_F_VIEWS |
//                        NTR_F_PROJ builds (ss_pixel_color with EXACT1 and PROJ) or, for the refinement, of the NTR_F_LIST |
//                        NTR_F_PROJ builds, then one pass per reflection depth, and refine_pixel between the two rounds;
//   emul_proj_vs_rays    the projected factor-1 pass next to given_ray_color of its own camera rays (render_rays_kernel):
//                        colour bits, bounce records and counters must be identical.
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

// the frame parameters enqueue_frame sets for a w x h frame at factor ss under projection (kind, param)
FrameDev proj_frame(const Scene &S, int w, int h, int ss, int kind, float param) {
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = ss;
    f.width = w * ss; f.height = h * ss;
    f.half_w = (float)f.width / 2.0f; f.half_h = (float)f.height / 2.0f;
    f.fovI = tanf(S.dev.fov / 2) / f.half_w;
    f.proj = kind;
    if (kind != NTR_PROJ_PERSPECTIVE) f.proj_k = projection_k(kind, param, f.half_w);
    f.x0 = 0; f.y0 = 0; f.win_w = w; f.win_h = h;
    f.tiles_x = (w + NTR_TILE - 1) / NTR_TILE; f.tiles_y = (h + NTR_TILE - 1) / NTR_TILE;
    f.tile_row_first = 0; f.tile_row_step = 1; f.out_rows = h;
    return f;
}

template <int DT>
void camera_rays_t(Scene &S, int w, int h, int kind, float param, float *origins, float *dirs) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = S.dev.dim;
    const FrameDev f = proj_frame(S, w, h, 1, kind, param);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            float o[CAP], dir[CAP];
            primary_ray<DT, true>(S.dev, S.cam, f, x, y, o, dir);
            const size_t i = (size_t)y * w + x;
            memcpy(origins + i * D, o, sizeof(float) * D);
            memcpy(dirs + i * D, dir, sizeof(float) * D);
        }
    }
}

// one round of bounce passes over queue (q, qp), adding into rgb
template <int DT, int FLAGS>
void bounce_rounds(Scene &S, std::vector<Bounce<DT>> &q, std::vector<uint32_t> &qp, float *rgb, Counters &cnt, MailboxStore &ms) {
    std::vector<Bounce<DT>> qn;
    std::vector<uint32_t> qpn;
    while (!q.empty()) {
        qn.clear(); qpn.clear();
        for (size_t i = 0; i < q.size(); ++i) {
            float acc[3] = {0, 0, 0};
            VecEmit<DT> emit{&qn, &qpn, qp[i]};
            ray_color<DT, FLAGS>(S.dev, true, q[i].o, q[i].d, q[i].depth, q[i].skip, q[i].w, acc, emit, cnt, nullptr, &ms);
            rgb[(size_t)qp[i] * 3] += acc[0]; rgb[(size_t)qp[i] * 3 + 1] += acc[1]; rgb[(size_t)qp[i] * 3 + 2] += acc[2];
        }
        q.swap(qn); qp.swap(qpn);
    }
}

template <int DT, int FLAGS>
void render_proj_t(Scene &S, int w, int h, int ss, float t, int kind, float param, float *rgb, unsigned char *mask,
                   unsigned long long *cnt_out) {
    const bool adaptive = ss > 1 && t >= 0;
    Counters cnt;
    std::vector<Bounce<DT>> q;
    std::vector<uint32_t> qp;
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    // the base pass: the views-PROJ build (at factor 1 for an adaptive frame)
    const FrameDev f = proj_frame(S, w, h, adaptive ? 1 : ss, kind, param);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            const uint32_t pix = (uint32_t)y * w + x;
            VecEmit<DT> emit{&q, &qp, pix};
            ss_pixel_color<DT, FLAGS, VecEmit<DT>, true, true>(S.dev, S.cam, f, x, y, rgb + (size_t)pix * 3, emit, cnt, &ms);
        }
    }
    bounce_rounds<DT, FLAGS>(S, q, qp, rgb, cnt, ms);
    uint64_t refined = 0;
    if (adaptive) {
        // classify_kernel over the whole frame (no halo), then the list pass at factor ss over the refined slots
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) mask[(size_t)y * w + x] = refine_pixel(f, rgb, x, y, t) ? 1 : 0;
        const FrameDev fr = proj_frame(S, w, h, ss, kind, param);
        for (int y = 0; y < h; ++y) {
            for (int x = 0; x < w; ++x) {
                const uint32_t pix = (uint32_t)y * w + x;
                if (!mask[pix]) continue;
                ++refined;
                VecEmit<DT> emit{&q, &qp, pix};
                ss_pixel_color<DT, FLAGS, VecEmit<DT>, false, true>(S.dev, S.cam, fr, x, y, rgb + (size_t)pix * 3, emit, cnt, &ms);
            }
        }
        bounce_rounds<DT, FLAGS>(S, q, qp, rgb, cnt, ms);
    }
    ms.detach();
    cnt_out[0] = adaptive ? (unsigned long long)w * h + refined * ss * ss : (unsigned long long)w * h * ss * ss;
    put_counters(cnt_out + 1, cnt);
}

template <int DT, int FLAGS>
void vs_rays_t(Scene &S, int w, int h, int kind, float param, float *rgb_frame, float *rgb_rays, float *origins, float *dirs,
               unsigned long long *cnt, unsigned long long *rec) {
    const int D = S.dev.dim;
    const FrameDev f = proj_frame(S, w, h, 1, kind, param);
    camera_rays_t<DT>(S, w, h, kind, param, origins, dirs);
    Counters c1, c2;
    std::vector<Bounce<DT>> q1, q2;
    std::vector<uint32_t> p1, p2;
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            const uint32_t pix = (uint32_t)y * w + x;
            VecEmit<DT> e1{&q1, &p1, pix};
            ss_pixel_color<DT, FLAGS, VecEmit<DT>, true, true>(S.dev, S.cam, f, x, y, rgb_frame + (size_t)pix * 3, e1, c1, &ms);
            VecEmit<DT> e2{&q2, &p2, pix};
            given_ray_color<DT, FLAGS>(S.dev, origins + (size_t)pix * D, dirs + (size_t)pix * D, rgb_rays + (size_t)pix * 3, e2, c2,
                                       &ms, (PrimaryAov<DT> *)nullptr);
        }
    }
    ms.detach();
    put_counters(cnt, c1);
    put_counters(cnt + 7, c2);
    rec[0] = q1.size(); rec[1] = q2.size();
    rec[2] = same_records<DT>(q1, q2, D) && p1 == p2;
}

}  // namespace

extern "C" {

// The w x h view's camera rays under projection (kind, param): origins / dirs w*h x D floats, ray y*w + x is pixel (x, y).
__attribute__((visibility("default"))) int emul_camera_rays(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                             int w, int h, int kind, float param, int force_generic,
                                                             float *origins, float *dirs) {
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT) camera_rays_t<DT>(S, w, h, kind, param, origins, dirs)
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

// A w x h frame at factor ss (1..NTR_MAX_SUPERSAMPLING) under projection (kind, param); threshold t >= 0 with ss > 1 makes it
// adaptive, and mask (w*h bytes) then receives the refine mask.  rgb: w*h*3 floats, counters: primary rays then the 7 words of
// emul_rays (reflection, shadow, node steps, simplex tests, solid tests, shaded hits, truncated).
__attribute__((visibility("default"))) int emul_render_proj(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                             int w, int h, int ss, float t, int kind, float param, int force_generic,
                                                             float *rgb, unsigned char *mask, unsigned long long *counters) {
    if (ss < 1 || ss > NTR_MAX_SUPERSAMPLING) return -1;
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                   \
    if (S.flags & NTR_F_GENERAL) render_proj_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, w, h, ss, t, kind, param, rgb, mask, counters); \
    else render_proj_t<DT, NTR_F_COUNT>(S, w, h, ss, t, kind, param, rgb, mask, counters)
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

// The projected factor-1 pass and given_ray_color of its camera rays (written to origins / dirs, w*h x D): rgb_frame /
// rgb_rays w*h*3 floats; counters 2 x 7 words, frame then rays; records: [0] frame count, [1] rays count, [2] 1 if identical.
__attribute__((visibility("default"))) int emul_proj_vs_rays(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                              int w, int h, int kind, float param, int force_generic,
                                                              float *rgb_frame, float *rgb_rays, float *origins, float *dirs,
                                                              unsigned long long *counters, unsigned long long *records) {
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                   \
    if (S.flags & NTR_F_GENERAL) vs_rays_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, w, h, kind, param, rgb_frame, rgb_rays, origins, dirs, counters, records); \
    else vs_rays_t<DT, NTR_F_COUNT>(S, w, h, kind, param, rgb_frame, rgb_rays, origins, dirs, counters, records)
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

}  // extern "C"
