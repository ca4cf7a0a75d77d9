// TEST INFRASTRUCTURE ONLY -- the primary pass of a batch of views at factor 1 against the plain primary pass, compiled into
// tests/host_emul/libhostemul_views.so (tests/emul_views_lib.py).  It builds on emul.cpp (scene setup, the emitter, the
// dimension dispatch), which is included whole, and adds one entry point.
//
// The NTR_F_VIEWS kernels trace every pixel with trace_core.cuh's ss_pixel_color at FrameDev::ss, factor 1 included
// (EXACT1 = true); the plain builds run primary_ray + box_color / ray_color.  At factor 1 both must give the same colour
// bits, bounce records and counters, for the frames of a batch of views to be those of ntr_render.
#include "emul.cpp"

namespace {

template <int DT>
bool same_records(const std::vector<Bounce<DT>> &a, const std::vector<Bounce<DT>> &b, int D) {
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i) {
        // the lanes past D are never read: compare the first D, bit for bit
        if (memcmp(a[i].o, b[i].o, sizeof(float) * D) || memcmp(a[i].d, b[i].d, sizeof(float) * D) ||
            memcmp(a[i].w, b[i].w, sizeof a[i].w) || a[i].skip.ref != b[i].skip.ref || a[i].skip.lane != b[i].skip.lane ||
            a[i].depth != b[i].depth)
            return false;
    }
    return true;
}

template <int DT, int FLAGS, bool EXACT1>
void compare_t(Scene &S, int w, int h, float *rgb_plain, float *rgb_views, unsigned long long *cnt, unsigned long long *rec) {
    constexpr int CAP = DimCap<DT>::value;
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
            primary_ray<DT>(S.dev, S.cam, f, x, y, o, dir);
            if (S.dev.kind == NTR_SCENE_BOX) box_color<DT>(S.dev, o, dir, acc, &prim);
            else {
                VecEmit<DT> emit{&q1, &p1, pix};
                ray_color<DT, FLAGS>(S.dev, true, o, dir, 0, none, one, acc, emit, c1, &prim, &ms);
            }
            rgb_plain[pix * 3] = acc[0]; rgb_plain[pix * 3 + 1] = acc[1]; rgb_plain[pix * 3 + 2] = acc[2];
            // the NTR_F_VIEWS builds
            VecEmit<DT> emit{&q2, &p2, pix};
            ss_pixel_color<DT, FLAGS, VecEmit<DT>, EXACT1>(S.dev, S.cam, f, x, y, rgb_views + (size_t)pix * 3, emit, c2, &ms);
        }
    }
    ms.detach();
    const Counters *c[2] = {&c1, &c2};
    for (int k = 0; k < 2; ++k) {
        unsigned long long *o = cnt + 7 * k;
        o[0] = c[k]->reflection_rays; o[1] = c[k]->shadow_rays; o[2] = c[k]->node_steps; o[3] = c[k]->simplex_tests;
        o[4] = c[k]->solid_tests; o[5] = c[k]->shaded_hits; o[6] = c[k]->truncated;
    }
    rec[0] = q1.size(); rec[1] = q2.size();
    rec[2] = same_records<DT>(q1, q2, S.dev.dim) && p1 == p2;
}

}  // namespace

extern "C" {

// A w x h frame at factor 1 both ways.  exact != 0: ss_pixel_color as the NTR_F_VIEWS kernels run it (EXACT1), 0: as the
// NTR_F_SS kernels do.  rgb_plain / rgb_views: w*h*3 floats; counters: 2 x 7 words (reflection, shadow, node steps, simplex
// tests, solid tests, shaded hits, truncated) plain then views; records: [0] plain count, [1] views count, [2] 1 if identical.
__attribute__((visibility("default"))) int emul_views_factor1(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                               int w, int h, int force_generic, int exact, float *rgb_plain,
                                                               float *rgb_views, unsigned long long *counters,
                                                               unsigned long long *records) {
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                           \
    if (exact) {                                                                                                           \
        if (S.flags & NTR_F_GENERAL) compare_t<DT, NTR_F_GENERAL | NTR_F_COUNT, true>(S, w, h, rgb_plain, rgb_views, counters, records); \
        else compare_t<DT, NTR_F_COUNT, true>(S, w, h, rgb_plain, rgb_views, counters, records);                        \
    } else {                                                                                                               \
        if (S.flags & NTR_F_GENERAL) compare_t<DT, NTR_F_GENERAL | NTR_F_COUNT, false>(S, w, h, rgb_plain, rgb_views, counters, records); \
        else compare_t<DT, NTR_F_COUNT, false>(S, w, h, rgb_plain, rgb_views, counters, records);                       \
    }
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

}  // extern "C"
