// TEST INFRASTRUCTURE ONLY -- the frame driver of emul.cpp for supersampled frames (ntr_scene_set_supersampling),
// compiled into tests/host_emul/libhostemul_ss.so (tests/emul_ss_lib.py).  It builds on emul.cpp (scene setup, the
// bounce-pass driver's emitter, the dimension dispatch), which is included whole, and adds one entry point.
//
// As in capi.cu's enqueue_frame, FrameDev describes the ss-times-larger view; the primary pass runs trace_core.cuh's
// ss_pixel_color for every output pixel -- the code the NTR_F_SS kernels inline -- and the bounce passes are emul.cpp's.
#include "emul.cpp"

namespace {

template <int DT, int FLAGS>
void render_ss_t(Scene &S, int w, int h, int ss, float *rgb, unsigned long long *cnt_out) {
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = ss;
    f.width = w * ss; f.height = h * ss;
    f.half_w = (float)f.width / 2.0f; f.half_h = (float)f.height / 2.0f;
    f.fovI = tanf(S.dev.fov / 2) / f.half_w;
    Counters cnt;
    std::vector<Bounce<DT>> q, qn;
    std::vector<uint32_t> qp, qpn;
    MailboxStore ms;
    ms.attach(S.dev.mb_table, S.dev.mb_words, S.dev.mb_threads, 0, S.dev.n_simplex, S.dev.mb_shift);
    for (int y = 0; y < h; ++y) {
        for (int x = 0; x < w; ++x) {
            const uint32_t pix = (uint32_t)y * w + x;
            VecEmit<DT> emit{&q, &qp, pix};
            ss_pixel_color<DT, FLAGS>(S.dev, S.cam, f, x, y, rgb + (size_t)pix * 3, emit, cnt, &ms);
        }
    }
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
    ms.detach();
    if (cnt_out) {
        cnt_out[0] = (unsigned long long)w * h * ss * ss; cnt_out[1] = cnt.reflection_rays; cnt_out[2] = cnt.shadow_rays;
        cnt_out[3] = cnt.node_steps; cnt_out[4] = cnt.simplex_tests; cnt_out[5] = cnt.solid_tests; cnt_out[6] = cnt.shaded_hits;
        cnt_out[7] = 0;
        cnt_out[8] = cnt.truncated;
    }
}

}  // namespace

extern "C" {

// A w x h frame with supersampling factor ss in 1..NTR_MAX_SUPERSAMPLING (anything else: -1); force_generic != 0 runs the
// run-time-dimension instantiation.  rgb: w*h*3 floats, counters: the 9 ntr_counters words.
__attribute__((visibility("default"))) int emul_render_ss(const ntr_scene_desc *d, const float *cam_origin,
                                                           const float *cam_axes, int w, int h, int ss, int force_generic,
                                                           float *rgb, unsigned long long *counters) {
    if (ss < 1 || ss > NTR_MAX_SUPERSAMPLING) return -1;
    Scene S;
    setup(S, d, cam_origin, cam_axes);
#define CALL(DT)                                                                                                  \
    if (S.flags & NTR_F_GENERAL) render_ss_t<DT, NTR_F_GENERAL | NTR_F_COUNT>(S, w, h, ss, rgb, counters);      \
    else render_ss_t<DT, NTR_F_COUNT>(S, w, h, ss, rgb, counters)
    DISPATCH_DIM(force_generic ? 0 : d->dim, CALL)
#undef CALL
    return 0;
}

}  // extern "C"
