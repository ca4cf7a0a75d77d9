// TEST INFRASTRUCTURE ONLY -- the AOV capture of the NTR_F_VIEWS | NTR_F_AOV kernels on the host, compiled into
// tests/host_emul/libhostemul_aov.so (tests/emul_aov_lib.py).  It builds on emul.cpp (scene setup, the emitter, the dimension
// dispatch), which is included whole, and adds two entry points.
//
// The AOV builds call trace_core.cuh's ss_pixel_color with a PrimaryAov: it must leave the colour bits, the emitted bounce
// records and the counters exactly as they are without it, and give the hit and shading normal of the pixel's plain primary ray.
#include "emul.cpp"

namespace {

template <int DT>
bool same_records_aov(const std::vector<Bounce<DT>> &a, const std::vector<Bounce<DT>> &b, int D) {
    if (a.size() != b.size()) return false;
    for (size_t i = 0; i < a.size(); ++i) {
        if (memcmp(a[i].o, b[i].o, sizeof(float) * D) || memcmp(a[i].d, b[i].d, sizeof(float) * D) ||
            memcmp(a[i].w, b[i].w, sizeof a[i].w) || a[i].skip.ref != b[i].skip.ref || a[i].skip.lane != b[i].skip.lane ||
            a[i].depth != b[i].depth)
            return false;
    }
    return true;
}

// the frame of the views kernels at factor ss (FrameDev as enqueue_frame fills it)
FrameDev views_frame(const Scene &S, int w, int h, int ss) {
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = ss;
    f.width = w * ss; f.height = h * ss;
    f.half_w = (float)f.width / 2.0f; f.half_h = (float)f.height / 2.0f;
    f.fovI = tanf(S.dev.fov / 2) / f.half_w;
    f.aov_half_w = (float)w / 2.0f; f.aov_half_h = (float)h / 2.0f;
    f.aov_fovI = tanf(S.dev.fov / 2) / f.aov_half_w;
    return f;
}

template <int DT, int FLAGS>
void aov_t(Scene &S, int w, int h, int ss, int32_t *ids, float *depth, float *normals, float *dirs, float *rgb_plain,
           float *rgb_aov, unsigned long long *cnt, unsigned long long *rec) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = S.dev.dim;
    const FrameDev f = views_frame(S, w, h, ss);
    Counters c1, c2;
    std::vector<Bounce<DT>> q1, q2;
    std::vector<uint32_t> p1, p2;
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            const uint32_t pix = (uint32_t)y * w + x;
            VecEmit<DT> e1{&q1, &p1, pix}, e2{&q2, &p2, pix};
            ss_pixel_color<DT, FLAGS, VecEmit<DT>, true>(S.dev, S.cam, f, x, y, rgb_plain + (size_t)pix * 3, e1, c1, &ms);
            PrimaryAov<DT> a;
            ss_pixel_color<DT, FLAGS, VecEmit<DT>, true>(S.dev, S.cam, f, x, y, rgb_aov + (size_t)pix * 3, e2, c2, &ms, &a);
            // what store_aov (kernels.cuh) writes
            const bool hit = a.hit.ref != NTR_NONE_REF;
            ids[pix] = !hit ? -1 : (S.dev.kind == NTR_SCENE_BOX ? 0 : flat_prim_id(S.dev, a.hit.ref, a.hit.lane));
            depth[pix] = a.hit.dist;
            for (int k = 0; k < D; ++k) normals[(size_t)pix * D + k] = a.n[k];
            float o[CAP], dir[CAP];
            primary_ray_of<DT>(S.dev, S.cam, f.aov_fovI, f.aov_half_w, f.aov_half_h, x, y, o, dir);
            for (int k = 0; k < D; ++k) dirs[(size_t)pix * D + k] = dir[k];
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
    rec[2] = same_records_aov<DT>(q1, q2, D) && p1 == p2;
}

}  // namespace

extern "C" {

// A w x h batch view at factor ss through ss_pixel_color as the NTR_F_VIEWS kernels run it, without and with the AOV capture.
// ids / depth: w*h, normals / dirs: w*h*dim (dirs: the plain primary ray of every pixel); rgb_plain / rgb_aov: w*h*3 floats;
// counters: 2 x 7 words (as emul_views_factor1) without then with; records: [0] / [1] counts, [2] 1 if identical.
__attribute__((visibility("default"))) int emul_aov_pass(const ntr_scene_desc *d, const float *cam_origin, const float *cam_axes,
                                                          int w, int h, int ss, int force_generic, int32_t *ids, float *depth,
                                                          float *normals, float *dirs, float *rgb_plain, float *rgb_aov,
                                                          unsigned long long *counters, unsigned long long *records) {
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                              \
    if (S.flags & NTR_F_GENERAL) aov_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, w, h, ss, ids, depth, normals, dirs, rgb_plain, rgb_aov, counters, records); \
    else aov_t<DT, NTR_F_COUNT>(S, w, h, ss, ids, depth, normals, dirs, rgb_plain, rgb_aov, counters, records);
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

// The pixels of a w x h view whose sample (0, 0) at factor ss is not the plain primary ray bit for bit (origin and direction),
// for the camera given and fov; 0 means ss_pixel_color may take the AOVs from that sample.
__attribute__((visibility("default"))) long long emul_aov_sample0_mismatches(int dim, const float *cam_origin, const float *cam_axes,
                                                                             float fov, int w, int h, int ss) {
    SceneDev s;
    memset(&s, 0, sizeof s);
    s.dim = dim; s.fov = fov;
    CameraDev cam;
    memset(&cam, 0, sizeof cam);
    for (int i = 0; i < dim; ++i) {
        cam.origin[i] = cam_origin[i];
        cam.right[i] = cam_axes[i]; cam.up[i] = cam_axes[dim + i]; cam.fwd[i] = cam_axes[2 * dim + i];
    }
    Scene S;
    S.dev = s;
    const FrameDev f = views_frame(S, w, h, ss);
    long long bad = 0;
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            float o1[NTR_MAXD], d1[NTR_MAXD], o2[NTR_MAXD], d2[NTR_MAXD];
            primary_ray<0>(s, cam, f, ss * x, ss * y, o1, d1);
            primary_ray_of<0>(s, cam, f.aov_fovI, f.aov_half_w, f.aov_half_h, x, y, o2, d2);
            bad += memcmp(o1, o2, sizeof(float) * dim) != 0 || memcmp(d1, d2, sizeof(float) * dim) != 0;
        }
    return bad;
}

}  // extern "C"
