// TEST INFRASTRUCTURE ONLY -- the refine rule of adaptive supersampling (ntr_scene_set_supersampling_threshold) and the
// accumulator-slot layout it reads, compiled for the host from ntracer_b200/csrc/trace_core.cuh into
// tests/host_emul/libhostemul_aa.so (tests/emul_aa_lib.py).  Nothing under ntracer_b200/ loads it.
//
// It fills the slots of one launch (its own pixels, then the halo) from a plain frame of the whole view, as the base and
// halo passes do on the device, and runs refine_pixel -- the function classify_kernel runs -- on every owned pixel.
#include <string.h>

#include <vector>

#include <vector_types.h>

#include "../../ntracer_b200/csrc/trace_core.cuh"

using namespace ntr;

extern "C" {

// view_rgb: vh x vw x 3 floats; window (x0, y0, win_w, win_h) of the view, tile rows trf, trf + trs, ... of it (compact:
// packed as a strip).  mask (win_h x win_w, window layout) receives the rule's result on the owned rows.  Returns the
// number of halo pixels traced.
__attribute__((visibility("default"))) long long emul_refine_mask(const float *view_rgb, int vw, int vh, int x0, int y0,
                                                                   int win_w, int win_h, int trf, int trs, int compact,
                                                                   float t, unsigned char *mask) {
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = 1; f.width = vw; f.height = vh;
    f.x0 = x0; f.y0 = y0; f.win_w = win_w; f.win_h = win_h;
    f.tiles_x = (win_w + NTR_TILE - 1) / NTR_TILE;
    f.tiles_y = (win_h + NTR_TILE - 1) / NTR_TILE;
    f.tile_row_first = trf; f.tile_row_step = trs; f.compact = compact;
    f.out_rows = compact ? owned_tile_rows(f) * NTR_TILE : win_h;
    const size_t npix = (size_t)win_w * f.out_rows, nhalo = halo_slots(f);
    // a slot nobody traced reads as a colour far from every real one: the rule would refine wherever it is read
    std::vector<float> acc((npix + nhalo) * 3, 1e30f);
    auto fill = [&](size_t slot, int wx, int wy) {
        const float *c = view_rgb + ((size_t)(y0 + wy) * vw + (x0 + wx)) * 3;
        acc[slot * 3] = c[0]; acc[slot * 3 + 1] = c[1]; acc[slot * 3 + 2] = c[2];
    };
    int r = 0, wx = 0, wy = 0;
    for (int out_row = 0; out_row < f.out_rows; ++out_row) {
        wy = window_row(f, out_row);
        if (owned_row(f, wy, &r))
            for (int x = 0; x < win_w; ++x) fill((size_t)out_row * win_w + x, x, wy);
    }
    long long traced = 0;
    for (size_t h = 0; h < nhalo; ++h)
        if (halo_pixel(f, (uint32_t)h, &wx, &wy)) { fill(npix + h, wx, wy); ++traced; }
    for (wy = 0; wy < win_h; ++wy) {
        if (!owned_row(f, wy, &r)) continue;
        for (wx = 0; wx < win_w; ++wx) mask[(size_t)wy * win_w + wx] = refine_pixel(f, acc.data(), wx, wy, t) ? 1 : 0;
    }
    return traced;
}

}  // extern "C"
