// kernels.cuh -- the __global__ kernels of the render path, templated on the dimension (DT = 3..8, 0 = run-time
// dimension) and the variant flags; instantiated per dimension in kern_d*.cu so the translation units
// compile in parallel.
//
//   render_pass_kernel  persistent warps; primary pass: atomic block queue over 32x32 tiles (reference
//                       worker_draw, src/render.cpp:468-493) + ray generation + traversal + shading + pixel
//                       packing epilogue; secondary passes: the same per-ray code over a wavefront queue of
//                       reflection bounces written by the previous pass with warp-aggregated atomics.
//   pack_kernel         float accumulator -> ImageFormat bytes (reference process_pixel, src/render.cpp:396-466)
//   trace_rays_kernel / occludes_rays_kernel   KDNode.intersects / KDNode.occludes parity hooks
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "trace_warp.cuh"

namespace ntr {

constexpr int kCtaThreads = 128;

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Deferred-ray sink: appends to the next pass's queue.  The slot index comes from ONE atomicAdd per
// converged group of lanes (ballot of the active mask + prefix popcount), not one per ray.
template <int DT> struct QueueEmit {
    const QueueDev &q;
    const ControlDev &ctl;
    uint32_t pixel;
    bool enabled;       // false: the frame needs no secondary passes (nothing reflective) -- drop the bounce
    __device__ __forceinline__ void operator()(const Bounce<DT> &b) const {
        if (!enabled) return;
        const unsigned mask = __activemask();
        const int leader = __ffs(mask) - 1;
        const int lane = threadIdx.x & 31;
        uint32_t base = 0;
        if (lane == leader) base = atomicAdd(q.out_count, (uint32_t)__popc(mask));
        base = __shfl_sync(mask, base, leader);
        const uint32_t idx = base + (uint32_t)__popc(mask & lanemask_lt());
        if (idx >= q.capacity) { *ctl.overflow = 1u; return; }
        float4 *rec = q.out + (size_t)idx * q.rec4;
        rec[0] = make_float4(__uint_as_float(pixel), __uint_as_float(b.skip.ref),
                             __int_as_float((b.skip.lane & 0xFFFF) | (b.depth << 16)), 0.0f);
        rec[1] = make_float4(b.w[0], b.w[1], b.w[2], 0.0f);
        constexpr int CAP = DimCap<DT>::value;
        const int D4 = (int)(q.rec4 - 2) / 2;       // float4s per vector
#pragma unroll
        for (int k = 0; k < (CAP + 3) / 4; ++k) {
            if (k < D4) {
                float4 vo, vd;
                vo.x = 4 * k + 0 < CAP ? b.o[4 * k + 0] : 0.f; vo.y = 4 * k + 1 < CAP ? b.o[4 * k + 1] : 0.f;
                vo.z = 4 * k + 2 < CAP ? b.o[4 * k + 2] : 0.f; vo.w = 4 * k + 3 < CAP ? b.o[4 * k + 3] : 0.f;
                vd.x = 4 * k + 0 < CAP ? b.d[4 * k + 0] : 0.f; vd.y = 4 * k + 1 < CAP ? b.d[4 * k + 1] : 0.f;
                vd.z = 4 * k + 2 < CAP ? b.d[4 * k + 2] : 0.f; vd.w = 4 * k + 3 < CAP ? b.d[4 * k + 3] : 0.f;
                rec[2 + k] = vo;
                rec[2 + D4 + k] = vd;
            }
        }
    }
};
struct NullEmit {
    template <typename B> __device__ __forceinline__ void operator()(const B &) const {}
};

__device__ __forceinline__ void flush_counters(const ControlDev &ctl, const Counters &cnt) {
    unsigned long long v[7] = {cnt.reflection_rays, cnt.shadow_rays, cnt.node_steps, cnt.simplex_tests,
                               cnt.solid_tests, cnt.shaded_hits, cnt.truncated};
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        unsigned long long x = v[k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, off);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(ctl.counters + 1 + k, x);     // slot 0 = primary_rays (host)
    }
}

// Warp-cooperative store of an 8x4 pixel block: pixels are staged in shared memory in memory byte order,
// then every lane moves one 16-byte chunk of one row segment with the widest aligned store.
// `packed`: the frame the block belongs to (f.packed, or frame v of a batch of views)
__device__ __forceinline__ void store_block_packed(const FrameDev &f, unsigned char *packed, unsigned char *stage /*512 B per warp*/,
                                                   int px0, int py0, int ncols, int nrows, int out_row0,
                                                   const uint32_t w[4], bool inside) {
    const int lane = threadIdx.x & 31;
    const int bpp = f.fmt.bytes_per_pixel;
    const int r = lane >> 3, c = lane & 7;
    if (inside) {
        unsigned char *d = stage + r * 128 + c * bpp;
        for (int j = 0; j < bpp; ++j) {
            const int sj = f.fmt.reversed ? bpp - 1 - j : j;
            d[j] = (unsigned char)(w[sj >> 2] >> (8 * (3 - (sj & 3))));
        }
    }
    __syncwarp();
    const int seg = ncols * bpp;
    if (r < nrows) {
        int off = c * 16;
        int n = seg - off;
        if (n > 16) n = 16;
        if (n > 0) {
            unsigned char *dst = packed + (size_t)(out_row0 + r) * f.fmt.pitch + (size_t)px0 * bpp + off;
            const unsigned char *src = stage + r * 128 + off;
            while (n > 0) {
                const size_t a = (size_t)dst | (size_t)src;      // both sides must be aligned for the unit
                if (n >= 16 && (a & 15) == 0) { *(uint4 *)dst = *(const uint4 *)src; dst += 16; src += 16; n -= 16; }
                else if (n >= 8 && (a & 7) == 0) { *(uint2 *)dst = *(const uint2 *)src; dst += 8; src += 8; n -= 8; }
                else if (n >= 4 && (a & 3) == 0) { *(uint32_t *)dst = *(const uint32_t *)src; dst += 4; src += 4; n -= 4; }
                else { *dst++ = *src++; --n; }
            }
        }
    }
    __syncwarp();
}

#ifndef NTR_MIN_CTAS
#define NTR_MIN_CTAS 8
#endif
#ifndef NTR_FETCH_STATS
#define NTR_FETCH_STATS 0          // diagnostic: per-fetch durations (see ControlDev::fetch_stats); never in the shipped build
#endif
// above 8 dimensions the ray alone (origin, direction, hit point) is 30+ registers: fewer CTAs per SM, more registers
#ifndef NTR_MIN_CTAS_HI
#define NTR_MIN_CTAS_HI 5          // measured on config 5 (16 k simplexes): 3 -> 31.7 ms, 4 -> 25.5, 5 -> 23.3, 6 -> 24.6, 8 -> 32.6
#endif
#ifndef NTR_MIN_CTAS_MID
#define NTR_MIN_CTAS_MID 6         // dimensions 6..8; measured on config 3 (6-D): 8 -> 0.550 ms, 6 -> 0.536 ms
#endif
// NTR_F_WIDE: measured on config 4 (call 25) with the whole 4-D family at 8 / 7 / 6 / 5 CTAs per SM: the full frame wants
// occupancy (42.6 / 43.6 / 45.5 / 47.4 ms) but its two last bounce passes (0.9 M and 0.6 M rays) and every pass of a 1/8
// share are decided by a few long rays and want registers (share: 15.2 / 14.9 / 15.0 / 14.4 ms), so both builds exist and
// the host picks per pass (capi.cu: wide_below).
#ifndef NTR_MIN_CTAS_WIDE
#define NTR_MIN_CTAS_WIDE 5
#endif
// NTR_F_LIST: the list-driven primary pass of an adaptively supersampled frame.  Every fetch takes up to 32 list entries,
// one accumulator slot per lane; the lane traces its pixel with ss_pixel_color at the factor f describes (1 for the halo,
// s for the refinement), stores the colour over the slot and emits the bounces for the next pass.
template <int DT, int FLAGS>
__device__ __forceinline__ void list_pass(const SceneDev &s, const CameraDev &cam, const FrameDev &f, const QueueDev &q,
                                          const ControlDev &ctl) {
    const int lane = threadIdx.x & 31;
    Counters cnt;
    MailboxStore ms;
    ms.attach((FLAGS & NTR_F_GENERAL) ? s.mb_table : nullptr, s.mb_words, s.mb_threads, blockIdx.x * blockDim.x + threadIdx.x, s.n_simplex, s.mb_shift);
    const uint32_t npix = (uint32_t)f.win_w * (uint32_t)f.out_rows;
    const uint32_t total = f.list_count ? *f.list_count : f.list_n;
    for (;;) {
        uint32_t b = 0;
        if (lane == 0) b = atomicAdd(ctl.tile_cursor, 32u);
        b = __shfl_sync(0xFFFFFFFFu, b, 0);
        if (b >= total) break;
        // the abort poll of the bounce passes: the fetch whose range crosses a multiple of 8192 entries looks
        if ((b & 8191u) < 32u && *ctl.abort_flag) {
            if (lane == 0) atomicAdd(ctl.tile_cursor, 0x40000000u);
            break;
        }
        const uint32_t idx = b + lane;
        uint32_t slot = 0;
        int wx = 0, wy = 0;
        bool inside = false;
        if (idx < total) {
            slot = f.list ? __ldg(f.list + idx) : npix + idx;
            if (slot < npix) {
                wx = (int)(slot % (uint32_t)f.win_w);
                wy = window_row(f, (int)(slot / (uint32_t)f.win_w));
                inside = true;
            } else {
                inside = halo_pixel(f, slot - npix, &wx, &wy);
            }
        }
        if (inside) {
            float acc[3];
            QueueEmit<DT> emit{q, ctl, slot, q.out != nullptr};
            ss_pixel_color<DT, FLAGS & (NTR_F_GENERAL | NTR_F_COUNT)>(s, cam, f, f.x0 + wx, f.y0 + wy, acc, emit, cnt, &ms);
            f.accum[(size_t)slot * 3 + 0] = acc[0]; f.accum[(size_t)slot * 3 + 1] = acc[1]; f.accum[(size_t)slot * 3 + 2] = acc[2];
        }
    }
    __syncwarp();
    ms.detach();
    flush_counters(ctl, cnt);
}

// The AOVs of pixel slot pix of a batch of views (NTR_F_AOV): what ntr_primary_hit_ids stores, and the hit's normal
template <int DT>
__device__ __forceinline__ void store_aov(const SceneDev &s, const FrameDev &f, uint32_t pix, const PrimaryAov<DT> &a) {
    const bool hit = a.hit.ref != NTR_NONE_REF;
    if (f.aov_ids) f.aov_ids[pix] = !hit ? -1 : (s.kind == NTR_SCENE_BOX ? 0 : flat_prim_id(s, a.hit.ref, a.hit.lane));
    if (f.aov_depth) f.aov_depth[pix] = a.hit.dist;
    if (f.aov_normals) {
        const int D = NTR_D(DT, s);
        float *n = f.aov_normals + (size_t)pix * D;
#pragma unroll
        for (int k = 0; k < DimCap<DT>::value; ++k)
            if (k < D) n[k] = a.n[k];
    }
}

template <int DT, int FLAGS = 0> struct MinCtas {
    static constexpr int value = (FLAGS & NTR_F_WIDE) ? NTR_MIN_CTAS_WIDE : DT > 8 ? NTR_MIN_CTAS_HI : (DT >= 6 ? NTR_MIN_CTAS_MID : NTR_MIN_CTAS);
};
template <int DT, int FLAGS>
__global__ void __launch_bounds__(kCtaThreads, MinCtas<DT, FLAGS>::value)
render_pass_kernel(const __grid_constant__ SceneDev s, const __grid_constant__ CameraDev cam,
                   const __grid_constant__ FrameDev f, const __grid_constant__ QueueDev q,
                   const __grid_constant__ ControlDev ctl) {
    if constexpr ((FLAGS & NTR_F_LIST) != 0) {
        list_pass<DT, FLAGS>(s, cam, f, q, ctl);
        return;
    }
    constexpr int CAP = DimCap<DT>::value;
    __shared__ __align__(16) unsigned char stage_all[(kCtaThreads / 32) * 512];
    __shared__ int done_all[kCtaThreads / 32];
    unsigned char *stage = stage_all + (threadIdx.x >> 5) * 512;
    int *done_ctr = done_all + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    Counters cnt;

    // One loop serves both kinds of pass so that the per-ray code (ray_color and everything it inlines) exists
    // exactly once in the kernel: only the work fetch and the epilogue differ.
    constexpr bool VIEWS = (FLAGS & NTR_F_VIEWS) != 0;
    const bool primary = (FLAGS & (NTR_F_SS | NTR_F_VIEWS)) != 0 || q.in == nullptr;   // NTR_F_SS / NTR_F_VIEWS builds only run primary passes
    const int my_rows = f.tile_row_first < f.tiles_y
                            ? (f.tiles_y - f.tile_row_first + f.tile_row_step - 1) / f.tile_row_step : 0;
    uint32_t total = (uint32_t)my_rows * (uint32_t)f.tiles_x * NTR_BLOCKS_PER_TILE;
    if constexpr (VIEWS) total *= f.n_views;
    const int D4 = (int)(q.rec4 - 2) / 2;
    if (!primary) {
        total = *q.in_count;
        if (total > q.capacity) total = q.capacity;
    }
    uint32_t fetches = 0;
    MailboxStore ms;                    // this thread's column of the exact mailbox (scenes with big leaves), if any
    ms.attach((FLAGS & NTR_F_GENERAL) ? s.mb_table : nullptr, s.mb_words, s.mb_threads, blockIdx.x * blockDim.x + threadIdx.x, s.n_simplex, s.mb_shift);
    for (;;) {
        // ---------------- fetch: an 8x4 pixel block of a tile (primary) or up to 32 queued bounces ----------------
        uint32_t b = 0, take = 32;
        if (lane == 0) {
            if (primary) b = atomicAdd(ctl.tile_cursor, 1u);
            else {
                if (q.ring_start) {
                    const uint32_t pos = *(volatile uint32_t *)q.in_cursor;         // a peek: good enough to pick the size
                    // Rays through the centre of the scene box walk the giant leaves of star polytopes and cost 10-90x the
                    // mean (tools/ray_cost_map.py); the heavy-first sort puts them in rings 0..2 at the front of the pass.
                    // Warps take fewer of them per fetch, so that the expensive rays of a pass run side by side in many
                    // warps instead of 32 to a warp in lockstep.
                    take = pos < __ldg(q.ring_start + 1) ? (q.fetch_sizes & 0xFFu) : pos < __ldg(q.ring_start + 2) ? ((q.fetch_sizes >> 8) & 0xFFu)
                           : pos < __ldg(q.ring_start + 3) ? ((q.fetch_sizes >> 16) & 0xFFu) : 32u;
                }
                b = atomicAdd(q.in_cursor, take);
            }
        }
        b = __shfl_sync(0xFFFFFFFFu, b, 0);
        take = __shfl_sync(0xFFFFFFFFu, take, 0);
        if (b >= total) break;
        // renderer::state poll (reference render.cpp:412).  The flag lives in mapped host memory, so only every
        // 512th block / every 64th fetch of a warp looks at it (ncu: at every 64th block the PCIe read was 2.9 % of all
        // stall samples); whoever sees it pushes the cursor past the end for everybody.
        ++fetches;
#if NTR_FETCH_STATS
        const long long fetch_t0 = clock64();
#endif
        // (bounce passes: the fetch whose range crosses a multiple of 8192 rays looks, whatever its size)
        if ((primary ? (b & 511u) == 0 : (b & 8191u) < take) && *ctl.abort_flag) {
            if (lane == 0) atomicAdd(primary ? ctl.tile_cursor : q.in_cursor, 0x40000000u);
            break;
        }
        float o[CAP], dir[CAP];
        float w[3] = {1.0f, 1.0f, 1.0f};
        float acc[3] = {0.f, 0.f, 0.f};
        Skip skip = {NTR_NONE_REF, 0};
        int depth = 0;
        uint32_t pix = 0, view = 0;
        bool active = false, inside = false;
        int bx = 0, by = 0, px = 0, out_row0 = 0;
        HitRec prim;
        prim.dist = 0; prim.ref = NTR_NONE_REF; prim.lane = -1;
        long long t_start = 0;
        uint32_t cost_tile = 0;
        if (primary) {
            // Longest-processing-time-first scheduling: tiles are handed out in the order of their measured cost
            // in the previous frame of this view (order_tiles_kernel), so the kernel's tail consists of the cheapest
            // blocks (background) instead of whatever happens to be last in row-major order.
            uint32_t slot = b / NTR_BLOCKS_PER_TILE;
            const uint32_t sub = b % NTR_BLOCKS_PER_TILE;
            // a batch of views: block b is sub-block `sub` of tile slot `slot` in view `view`, tile-major with the views inner,
            // so the 32 blocks of a tile in every view are handed out together, in the tile order of the schedule
            // (view-major order, each view's tiles after the previous view's, measured 6.5 % slower on c4: DESIGN section 9)
            if constexpr (VIEWS) { view = slot % f.n_views; slot /= f.n_views; }
            const uint32_t tile = f.tile_order ? __ldg(f.tile_order + slot) : slot;
            cost_tile = tile;
            if (f.tile_cost) t_start = clock64();
            const int tyi = (int)(tile / (uint32_t)f.tiles_x), tx = (int)(tile % (uint32_t)f.tiles_x);
            const int ty = f.tile_row_first + tyi * f.tile_row_step;
            bx = tx * NTR_TILE + (int)(sub % (NTR_TILE / NTR_BLK_W)) * NTR_BLK_W;       // window coordinates
            by = ty * NTR_TILE + (int)(sub / (NTR_TILE / NTR_BLK_W)) * NTR_BLK_H;
            if (bx >= f.win_w || by >= f.win_h) continue;
            px = bx + (lane & 7);
            const int py = by + (lane >> 3);
            inside = px < f.win_w && py < f.win_h;
            // output row of the block: frame position, or the compacted strip of this rank
            out_row0 = f.compact ? (tyi * NTR_TILE + (by - ty * NTR_TILE)) : by;
            pix = (uint32_t)(out_row0 + (lane >> 3)) * (uint32_t)f.win_w + (uint32_t)px;
            if constexpr (VIEWS) pix += view * ((uint32_t)f.win_w * (uint32_t)f.out_rows);
            if (inside) {
                if constexpr (VIEWS) {
                    // the view's camera is read from global memory where it is used (by reference), not copied to registers;
                    // at factor 1 the pixel gets the plain path's bits (ss_pixel_color, EXACT1)
                    QueueEmit<DT> emit{q, ctl, pix, f.out_mode == NTR_OUT_ACCUM};
                    if constexpr ((FLAGS & NTR_F_AOV) != 0) {
                        PrimaryAov<DT> aov;
                        ss_pixel_color<DT, FLAGS & (NTR_F_GENERAL | NTR_F_COUNT), QueueEmit<DT>, true>(s, f.views[view], f, f.x0 + px, f.y0 + py,
                                                                                                        acc, emit, cnt, &ms, &aov);
                        store_aov<DT>(s, f, pix, aov);
                    } else {
                        ss_pixel_color<DT, FLAGS & (NTR_F_GENERAL | NTR_F_COUNT), QueueEmit<DT>, true>(s, f.views[view], f, f.x0 + px, f.y0 + py,
                                                                                                        acc, emit, cnt, &ms);
                    }
                } else if constexpr ((FLAGS & NTR_F_SS) != 0) {
                    // supersampled frame: the lane traces the ss x ss samples of its pixel right here, one after the other
                    // (the loop count is the same for every lane); their bounces go to the next pass already weighted
                    QueueEmit<DT> emit{q, ctl, pix, f.out_mode == NTR_OUT_ACCUM};
                    ss_pixel_color<DT, FLAGS & (NTR_F_GENERAL | NTR_F_COUNT)>(s, cam, f, f.x0 + px, f.y0 + py, acc, emit, cnt, &ms);
                } else {
                    primary_ray<DT>(s, cam, f, f.x0 + px, f.y0 + py, o, dir);
                    if (s.kind == NTR_SCENE_BOX) box_color<DT>(s, o, dir, acc, &prim);
                    else active = true;
                }
            }
        } else {
            const uint32_t idx = b + lane;
            if ((uint32_t)lane < take && idx < total) {
                const float4 *rec = q.in + (size_t)((q.in_perm && idx < q.n_sorted) ? __ldg(q.in_perm + idx) : idx) * q.rec4;
                const float4 h = rec[0], wv = rec[1];
                pix = __float_as_uint(h.x);
                skip.ref = __float_as_uint(h.y);
                const int ld = __float_as_int(h.z);
                skip.lane = (int)(short)(ld & 0xFFFF);
                depth = ld >> 16;
                w[0] = wv.x; w[1] = wv.y; w[2] = wv.z;
#pragma unroll
                for (int k = 0; k < (CAP + 3) / 4; ++k) {
                    if (k < D4) {
                        const float4 vo = rec[2 + k], vd = rec[2 + D4 + k];
                        if (4 * k + 0 < CAP) { o[4 * k + 0] = vo.x; dir[4 * k + 0] = vd.x; }
                        if (4 * k + 1 < CAP) { o[4 * k + 1] = vo.y; dir[4 * k + 1] = vd.y; }
                        if (4 * k + 2 < CAP) { o[4 * k + 2] = vo.z; dir[4 * k + 2] = vd.z; }
                        if (4 * k + 3 < CAP) { o[4 * k + 3] = vo.w; dir[4 * k + 3] = vd.w; }
                    }
                }
                active = true;
            }
        }
        // ---------------- the per-ray path ----------------
        // Two forms of the same algorithm (FLAGS & NTR_F_WARP, chosen by the host per scene).  Every lane for itself
        // (trace_core.cuh) is the faster one on ordinary trees: ncu, config 2: the warp form spends 17x the local-memory
        // traffic and twice the instruction-fetch stalls (profiles/r02_c2_warp_vs_lane_ncu_summary.txt).  The
        // warp-synchronous form (trace_warp.cuh: all 32 lanes enter, `active` says who has a ray; rays park at big leaves
        // and the warp splits them over its lanes when enough lanes are idle) wins where single rays walk leaves of
        // hundreds of items (config 4: 58.4 -> 49.9 ms, its 1/8-frame share 26.3 -> 19.9 ms).
        constexpr int RF = FLAGS & ~(NTR_F_WARP | NTR_F_WIDE | NTR_F_SS | NTR_F_VIEWS | NTR_F_AOV);      // the per-ray code knows nothing of the switches
        if constexpr ((FLAGS & NTR_F_WARP) != 0) {
            if (s.kind != NTR_SCENE_BOX) {          // warp-uniform
                if (!active) {
#pragma unroll
                    for (int k = 0; k < CAP; ++k) { o[k] = 0.0f; dir[k] = 1.0f; }
                }
                QueueEmit<DT> emit{q, ctl, pix, !primary || f.out_mode == NTR_OUT_ACCUM};
                ray_color_warp<DT, RF>(s, active, o, dir, depth, skip, w, acc, emit, cnt, &prim, done_ctr, &ms);
            }
        } else if ((FLAGS & (NTR_F_SS | NTR_F_VIEWS)) == 0 && active) {
            QueueEmit<DT> emit{q, ctl, pix, !primary || f.out_mode == NTR_OUT_ACCUM};
            ray_color<DT, RF>(s, active, o, dir, depth, skip, w, acc, emit, cnt, &prim, &ms);
        }
        if (primary && f.tile_cost && lane == 0) atomicAdd(f.tile_cost + cost_tile, (unsigned long long)(clock64() - t_start));
#if NTR_FETCH_STATS
        if (lane == 0 && ctl.fetch_stats) {
            const unsigned long long dt = (unsigned long long)(clock64() - fetch_t0);
            atomicMax(ctl.fetch_stats, dt);
            atomicAdd(ctl.fetch_stats + 1, dt);
            atomicAdd(ctl.fetch_stats + 2, 1ull);
            atomicAdd(ctl.fetch_stats + 8 + (63 - __clzll((long long)(dt | 1ull))), 1ull);
        }
#endif
        // ---------------- epilogue ----------------
        if (!primary) {
            if (active) {
                atomicAdd(f.accum + (size_t)pix * 3 + 0, acc[0]);
                atomicAdd(f.accum + (size_t)pix * 3 + 1, acc[1]);
                atomicAdd(f.accum + (size_t)pix * 3 + 2, acc[2]);
            }
            continue;
        }
        __syncwarp();
        if (f.out_mode == NTR_OUT_PACKED) {
            uint32_t pw[4] = {0, 0, 0, 0};
            if (inside) pack_pixel(f.fmt, acc, pw);
            const int ncols = min(NTR_BLK_W, f.win_w - bx), nrows = min(NTR_BLK_H, f.win_h - by);
            unsigned char *packed = f.packed;
            if constexpr (VIEWS) packed += (size_t)view * (size_t)f.fmt.pitch * (size_t)f.win_h;
            store_block_packed(f, packed, stage, bx, by, ncols, nrows, out_row0, pw, inside);
        } else if (inside) {
            if (f.out_mode == NTR_OUT_ACCUM) {
                f.accum[(size_t)pix * 3 + 0] = acc[0]; f.accum[(size_t)pix * 3 + 1] = acc[1]; f.accum[(size_t)pix * 3 + 2] = acc[2];
            } else {
                f.ids[pix] = prim.ref == NTR_NONE_REF ? -1 : (s.kind == NTR_SCENE_BOX ? 0 : flat_prim_id(s, prim.ref, prim.lane));
                if (f.dists) f.dists[pix] = prim.dist;
            }
        }
    }
    __syncwarp();
    ms.detach();
    flush_counters(ctl, cnt);
}

// Next frame's tile schedule: tiles sorted by decreasing cost (rank by counting; n <= a few thousand tiles), costs
// halved so that the schedule follows a moving camera with some inertia.
static __global__ void order_tiles_kernel(unsigned long long *cost, uint32_t *order, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const unsigned long long ci = cost[i];
        uint32_t rank = 0;
        for (uint32_t j = 0; j < n; ++j) {
            const unsigned long long cj = cost[j];
            rank += (cj > ci) || (cj == ci && j < i);
        }
        order[rank] = i;
    }
}
static __global__ void decay_tile_cost_kernel(unsigned long long *cost, uint32_t n) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) cost[i] >>= 1;
}

// KDNode.intersects for a batch of rays (reference src/ntracer_body.hpp:1412-1458)
template <int DT, int FLAGS>
__global__ void __launch_bounds__(kCtaThreads)
trace_rays_kernel(const __grid_constant__ SceneDev s, uint32_t n, const float *origins, const float *dirs,
                  float t_near, float t_far, const uint32_t *skip_ref, const int32_t *skip_lane, int32_t *ids,
                  float *dist, int32_t *ntrans, int32_t *hit_ids, float *hit_dists, int max_hits) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = NTR_D(DT, s);
    MailboxStore ms;
    ms.attach((FLAGS & NTR_F_GENERAL) ? s.mb_table : nullptr, s.mb_words, s.mb_threads, blockIdx.x * blockDim.x + threadIdx.x, s.n_simplex, s.mb_shift);
    // grid-stride: the host never launches more threads than the mailbox table has columns
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float o[CAP], dir[CAP];
#pragma unroll
        for (int k = 0; k < D; ++k) { o[k] = origins[(size_t)i * D + k]; dir[k] = dirs[(size_t)i * D + k]; }
        Skip skip = {skip_ref ? skip_ref[i] : NTR_NONE_REF, skip_lane ? skip_lane[i] : -1};
        GenState<DT> g;
        g.mb.big = ms.col ? &ms : nullptr;
        g.th.clear();
        HitRec oh;
        oh.dist = FLT_MAX; oh.ref = NTR_NONE_REF; oh.lane = -1;
        Counters cnt;
        const bool hit = trace_nearest<DT, FLAGS>(s, o, dir, skip, t_near, t_far, oh, &g, cnt);
        ids[i] = hit ? flat_prim_id(s, oh.ref, oh.lane) : -1;
        if (dist) dist[i] = hit ? oh.dist : 0.0f;
        if (ntrans) ntrans[i] = (FLAGS & NTR_F_GENERAL) ? g.th.n : 0;
        // the surviving transparent hits in the order the reference's list holds them (kdnode_intersects returns them
        // before the opaque hit, src/ntracer_body.hpp:1438-1456)
        if ((FLAGS & NTR_F_GENERAL) && hit_ids) {
            for (int k = 0; k < g.th.n && k < max_hits; ++k) {
                hit_ids[(size_t)i * max_hits + k] = flat_prim_id(s, g.th.ref[k], g.th.lane[k]);
                if (hit_dists) hit_dists[(size_t)i * max_hits + k] = g.th.dist[k];
            }
        }
    }
    ms.detach();
}

// KDNode.occludes (reference src/ntracer_body.hpp:1460-1496)
template <int DT, int FLAGS>
__global__ void __launch_bounds__(kCtaThreads)
occludes_rays_kernel(const __grid_constant__ SceneDev s, uint32_t n, const float *origins, const float *dirs,
                     const float *distance, const uint32_t *skip_ref, const int32_t *skip_lane, int32_t *occ,
                     int32_t *ntrans) {
    constexpr int CAP = DimCap<DT>::value;
    const int D = NTR_D(DT, s);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float o[CAP], dir[CAP];
#pragma unroll
    for (int k = 0; k < D; ++k) { o[k] = origins[(size_t)i * D + k]; dir[k] = dirs[(size_t)i * D + k]; }
    Skip skip = {skip_ref ? skip_ref[i] : NTR_NONE_REF, skip_lane ? skip_lane[i] : -1};
    HitList hits;
    hits.clear();
    Counters cnt;
    const bool r = trace_occludes<DT, FLAGS>(s, o, dir, distance ? distance[i] : FLT_MAX, skip, -FLT_MAX, FLT_MAX,
                                            &hits, cnt);
    occ[i] = r ? 1 : 0;
    if (ntrans) ntrans[i] = (!r && (FLAGS & NTR_F_GENERAL)) ? hits.n : 0;
}

// ---- launch table -------------------------------------------------------------------------------------
struct KernelSet {
    void (*render_pass)(dim3, dim3, cudaStream_t, const SceneDev &, const CameraDev &, const FrameDev &,
                        const QueueDev &, const ControlDev &);
    void (*trace_rays)(dim3, dim3, cudaStream_t, const SceneDev &, uint32_t, const float *, const float *, float,
                       float, const uint32_t *, const int32_t *, int32_t *, float *, int32_t *, int32_t *, float *, int);
    void (*occludes_rays)(dim3, dim3, cudaStream_t, const SceneDev &, uint32_t, const float *, const float *,
                          const float *, const uint32_t *, const int32_t *, int32_t *, int32_t *);
    int (*max_blocks_per_sm)();
};

template <int DT, int FLAGS> struct Launch {
    static void render_pass(dim3 g, dim3 b, cudaStream_t st, const SceneDev &s, const CameraDev &cam,
                            const FrameDev &f, const QueueDev &q, const ControlDev &ctl) {
        // NTR_LAUNCH_LOG=1: one line per launch naming the build that runs (family: the dimension, 0 = run-time dimension)
        const char *log = getenv("NTR_LAUNCH_LOG");
        if (log && atoi(log) != 0) fprintf(stderr, "ntr launch family=%d flags=%d grid=%u\n", DT, FLAGS, g.x);
        render_pass_kernel<DT, FLAGS><<<g, b, 0, st>>>(s, cam, f, q, ctl);
    }
    static void trace_rays(dim3 g, dim3 b, cudaStream_t st, const SceneDev &s, uint32_t n, const float *o,
                           const float *d, float tn, float tf, const uint32_t *sr, const int32_t *sl, int32_t *ids,
                           float *dist, int32_t *nt, int32_t *hit_ids, float *hit_dists, int max_hits) {
        trace_rays_kernel<DT, FLAGS><<<g, b, 0, st>>>(s, n, o, d, tn, tf, sr, sl, ids, dist, nt, hit_ids, hit_dists, max_hits);
    }
    static void occludes_rays(dim3 g, dim3 b, cudaStream_t st, const SceneDev &s, uint32_t n, const float *o,
                              const float *d, const float *ld, const uint32_t *sr, const int32_t *sl, int32_t *occ,
                              int32_t *nt) {
        occludes_rays_kernel<DT, FLAGS><<<g, b, 0, st>>>(s, n, o, d, ld, sr, sl, occ, nt);
    }
    static int max_blocks_per_sm() {
        int n = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, render_pass_kernel<DT, FLAGS>, kCtaThreads, 0);
        return n;
    }
    // the ray hooks have no warp form: both render variants share them
    static KernelSet get() {
        return KernelSet{&render_pass, &Launch<DT, FLAGS & 3>::trace_rays, &Launch<DT, FLAGS & 3>::occludes_rays, &max_blocks_per_sm};
    }
};

// defined in kern_d*.cu: variant index = FLAGS (0..255; NTR_F_WIDE builds exist for the general variant in 3..5 dimensions,
// everywhere else the index falls back to the build without it; NTR_F_SS, NTR_F_LIST and NTR_F_VIEWS builds exist in the
// per-lane, non-wide form only, so they override NTR_F_WARP and NTR_F_WIDE; NTR_F_AOV builds exist with NTR_F_VIEWS only)
const KernelSet *kernel_set_d3(int flags);
const KernelSet *kernel_set_d4(int flags);
const KernelSet *kernel_set_d5(int flags);
const KernelSet *kernel_set_d6(int flags);
const KernelSet *kernel_set_d7(int flags);
const KernelSet *kernel_set_d8(int flags);
const KernelSet *kernel_set_d9(int flags);
const KernelSet *kernel_set_d10(int flags);
const KernelSet *kernel_set_dn(int flags);

#define NTR_SS_SETS(DT)                                                                                 \
        static const KernelSet ss[4] = {Launch<DT, NTR_F_SS>::get(), Launch<DT, 1 | NTR_F_SS>::get(),   \
                                        Launch<DT, 2 | NTR_F_SS>::get(), Launch<DT, 3 | NTR_F_SS>::get()}; \
        if (flags & NTR_F_SS) return &ss[flags & 3];                                                     \
        static const KernelSet list[4] = {Launch<DT, NTR_F_LIST>::get(), Launch<DT, 1 | NTR_F_LIST>::get(), \
                                          Launch<DT, 2 | NTR_F_LIST>::get(), Launch<DT, 3 | NTR_F_LIST>::get()}; \
        if (flags & NTR_F_LIST) return &list[flags & 3];                                                 \
        static const KernelSet views[4] = {Launch<DT, NTR_F_VIEWS>::get(), Launch<DT, 1 | NTR_F_VIEWS>::get(), \
                                           Launch<DT, 2 | NTR_F_VIEWS>::get(), Launch<DT, 3 | NTR_F_VIEWS>::get()}; \
        static const KernelSet aovs[4] = {Launch<DT, NTR_F_VIEWS | NTR_F_AOV>::get(), Launch<DT, 1 | NTR_F_VIEWS | NTR_F_AOV>::get(), \
                                          Launch<DT, 2 | NTR_F_VIEWS | NTR_F_AOV>::get(), Launch<DT, 3 | NTR_F_VIEWS | NTR_F_AOV>::get()}; \
        if (flags & NTR_F_VIEWS) return (flags & NTR_F_AOV) ? &aovs[flags & 3] : &views[flags & 3];
#define NTR_INSTANTIATE_DIM(NAME, DT)                                                                  \
    const KernelSet *NAME(int flags) {                                                                  \
        NTR_SS_SETS(DT)                                                                                 \
        static const KernelSet sets[8] = {Launch<DT, 0>::get(), Launch<DT, 1>::get(), Launch<DT, 2>::get(), \
                                          Launch<DT, 3>::get(), Launch<DT, 4>::get(), Launch<DT, 5>::get(), \
                                          Launch<DT, 6>::get(), Launch<DT, 7>::get()};                  \
        return &sets[flags & 7];                                                                        \
    }
#define NTR_INSTANTIATE_DIM_WIDE(NAME, DT)                                                              \
    const KernelSet *NAME(int flags) {                                                                  \
        NTR_SS_SETS(DT)                                                                                 \
        static const KernelSet sets[8] = {Launch<DT, 0>::get(), Launch<DT, 1>::get(), Launch<DT, 2>::get(), \
                                          Launch<DT, 3>::get(), Launch<DT, 4>::get(), Launch<DT, 5>::get(), \
                                          Launch<DT, 6>::get(), Launch<DT, 7>::get()};                  \
        static const KernelSet wide[4] = {Launch<DT, 1 | NTR_F_WIDE>::get(), Launch<DT, 3 | NTR_F_WIDE>::get(), \
                                          Launch<DT, 5 | NTR_F_WIDE>::get(), Launch<DT, 7 | NTR_F_WIDE>::get()}; \
        if ((flags & NTR_F_WIDE) && (flags & NTR_F_GENERAL)) return &wide[(flags & 7) >> 1];          \
        return &sets[flags & 7];                                                                        \
    }

}  // namespace ntr
