// Plain-old-data types shared by the host side (arena builder, C ABI) and the device code.
// Layouts are described in DESIGN.md section 3 ("data layout in HBM").
#pragma once
#include <stdint.h>
#include <vector_types.h>   // uint4 / float4 (plain C++ header of the CUDA toolkit)

#include "../../include/ntracer_b200.h"

#define NTR_MAXD NTR_MAX_DIM
#define NTR_NONE_REF 0xFFFFFFFFu
#define NTR_IDX_MASK 0x3FFFFFFFu
#define NTR_TILE 32                 // RENDER_CHUNK_SIZE, reference src/render.cpp:43
#define NTR_BLK_W 8                 // one warp renders an 8x4 pixel block
#define NTR_BLK_H 4
#define NTR_BLOCKS_PER_TILE ((NTR_TILE / NTR_BLK_W) * (NTR_TILE / NTR_BLK_H))

#define NTR_THITS_CAP 16            // transparent hits kept per ray (reference is defined up to 10, tracer.hpp:26)
#define NTR_MAILBOX_CAP 40          // mailbox entries kept per traversal (reference is defined up to 20, tracer.hpp:27)
#define NTR_MAILBOX_SLOTS 64        // open-addressing table that holds them (trace_core.cuh: Mailbox)
// Scenes whose leaves are bigger than that table get an EXACT mailbox instead: one bit per leaf item and traversing
// thread, in a scene-wide table in device memory (trace_core.cuh: MailboxStore).  Up to this many items (simplexes +
// solids); bigger scenes keep the bounded table.
#define NTR_MAILBOX_MAX_KEYS 65536
#define NTR_MAILBOX_BITS_PER_WORD 24   // a word = generation tag (8 bits) | 24 item bits
#define NTR_STACK_CAP (NTR_MAX_TREE_DEPTH + 2)

// meta word stored in the last float slot of every simplex / solid record
#define NTR_META_OPAQUE 0x80000000u

// kernel variant flags (template parameter)
enum : int {
    NTR_F_GENERAL = 1,      // scene has transparent materials and/or solids: mailbox, transparent-hit list,
                            // explicit normal mirroring (reference quirks, DESIGN.md section 4)
    NTR_F_COUNT = 2,        // instrumented: node/primitive counters (never used for timing)
    NTR_F_WARP = 4,         // render_pass_kernel only: the warp-synchronous per-ray path (trace_warp.cuh), chosen for scenes
                            // with big leaves; otherwise every lane traces for itself (trace_core.cuh)
    NTR_F_WIDE = 8,         // render_pass_kernel only, general variant in 3..5 dimensions: 96 registers / 5 CTAs per SM instead of
                            // 64 / 8 -- no spills, fewer warps: the build for passes that end in a few long rays (kernels.cuh)
    NTR_F_SS = 16,          // render_pass_kernel only, per-lane form: the primary pass of a supersampled frame (FrameDev::ss > 1),
                            // every lane traces the ss x ss samples of its pixel one after the other (trace_core.cuh: ss_pixel_color)
    NTR_F_LIST = 32,        // render_pass_kernel only, per-lane form: the list-driven primary pass of an adaptively supersampled
                            // frame (FrameDev::list): every lane traces one listed pixel with ss_pixel_color at factor FrameDev::ss
    NTR_F_VIEWS = 64,       // render_pass_kernel only, per-lane form: the primary pass of a batch of views (ntr_render_views,
                            // FrameDev::views): the blocks of all views in one launch, every lane traces its pixel with
                            // ss_pixel_color at factor FrameDev::ss (1 included) through the camera of its view
    NTR_F_AOV = 128         // with NTR_F_VIEWS only: the lane also stores the hit id, depth and normal of its pixel's plain
                            // (factor-1) primary ray into FrameDev::aov_* (ntr_render_views_aovs)
};

struct SceneDev {
    const uint4 *nodes;             // ntr_node, 16 B
    const uint2 *leaf_items;        // {leaf ref (identity: (type<<30)|index), float offset of the item's record}
    const float *simplex;           // stride sstride floats: fn[D], d, p1[D], edges[D-1][D], pad.., meta
    const float *batches;           // batch blocks (see arena_pack.h): SoA plane part + per-lane edge parts + metas
    const float *solids;            // stride solstride floats: type, inv_orientation[D*D], position[D], orientation[D*D], pad.., meta
    const float *materials;         // 12 floats per material (10 used)
    const float *point_lights;      // stride D+3
    const float *global_lights;     // stride D+3
    uint32_t *mb_table;             // exact mailbox: mb_words words per thread, word w of thread t at [w * mb_threads + t] (nullptr: none)
    uint32_t mb_words, mb_threads;
    uint32_t mb_shift;              // mailbox key of a simplex / batch item = record index >> mb_shift (2 when the leaf items' record
                                    // indices stay distinct after dropping two bits: a tree of aligned 4-lane batches), solids follow
    uint32_t root;
    uint32_t n_simplex;
    int dim, batch, sstride, solstride;
    int lane_part;                  // floats per lane in a batch block's stage-2 part: D*D rounded up to 4
    int kind;
    int n_point, n_global;
    int shadows, camera_light, max_depth, bg_axis;
    float fov;
    float ambient[3], bg1[3], bg2[3], bg3[3];
    float bmin[NTR_MAXD], bmax[NTR_MAXD];
};

struct CameraDev {
    float origin[NTR_MAXD], right[NTR_MAXD], up[NTR_MAXD], fwd[NTR_MAXD];
};

struct FormatDev {
    int n_channels, bytes_per_pixel, reversed, pitch;
    float f_r[NTR_MAX_CHANNELS], f_g[NTR_MAX_CHANNELS], f_b[NTR_MAX_CHANNELS], f_c[NTR_MAX_CHANNELS];
    unsigned char bits[NTR_MAX_CHANNELS], tfloat[NTR_MAX_CHANNELS];
};

// What a render pass writes.
enum : int {
    NTR_OUT_PACKED = 0,     // pack straight into the image format (no secondary passes needed)
    NTR_OUT_ACCUM = 1,      // float RGB accumulator (secondary passes add to it, a pack kernel follows)
    NTR_OUT_IDS = 2         // primary hit ids + distances (parity hook)
};

struct FrameDev {
    int width, height;              // view size
    float half_w, half_h, fovI;     // flat_origin_ray_source, reference src/tracer.hpp:60-69
    int x0, y0;                     // window origin (calculate_color renders a 1x1 window)
    int win_w, win_h;               // window size in pixels
    int tiles_x, tiles_y;           // window size in 32x32 tiles
    int tile_row_first, tile_row_step, compact;   // multi-GPU interleave (tile rows ty % step == first)
    int out_rows;                   // rows of the output / accumulator: win_h, or owned tile rows * 32 when compact
    int out_mode;
    const uint32_t *tile_order;     // cost-sorted tile schedule of the primary pass (nullptr = row-major)
    unsigned long long *tile_cost;  // per owned tile: SM cycles spent on it this frame (feeds the next frame's order)
    unsigned char *packed;          // NTR_OUT_PACKED destination (device)
    float *accum;                   // NTR_OUT_ACCUM: 3 floats per window pixel
    int32_t *ids;                   // NTR_OUT_IDS
    float *dists;
    FormatDev fmt;
    int ss;                         // supersampling factor: width / height / half_w / half_h / fovI describe the ss-times-larger
                                    // view, the window and tile grid stay in output pixels (1: plain frame)
    // adaptive supersampling (ntr_scene_set_supersampling_threshold): the NTR_F_LIST pass traces the accumulator slots
    // list[0 .. *list_count) (list == nullptr: the halo slots npix .. npix + list_n, trace_core.cuh: halo_pixel)
    const uint32_t *list;
    const uint32_t *list_count;
    uint32_t list_n;
    // a batch of views (NTR_F_VIEWS): view v traces through views[v]; its pixels take accumulator slots and bounce-record pixel
    // words v * npix + pix (npix = win_w * out_rows), and its packed frame starts at packed + v * pitch * win_h
    const CameraDev *views;
    uint32_t n_views;
    // AOVs of a batch of views (NTR_F_AOV), per pixel slot v * npix + pix, nullptr where not wanted: the flat id of the plain
    // primary ray's opaque hit (-1: miss), its distance, and dim floats of the hit's normal.  aov_half_w / aov_half_h /
    // aov_fovI describe the plain (factor-1) view, whose ray a factor that is not a power of two traces separately.
    int32_t *aov_ids;
    float *aov_depth;
    float *aov_normals;
    float aov_half_w, aov_half_h, aov_fovI;
};

// One deferred ray of the wavefront (a reflection bounce): 16-byte aligned record.
// layout: [0] pixel, [1] skip_ref, [2] skip_lane | depth<<16, [3] pad, [4..6] weight rgb, [7] pad,
//         then origin[Dq], dir[Dq] with Dq = D rounded up to 4
struct QueueDev {
    float4 *in;                     // rays of this pass (nullptr for the primary pass)
    float4 *out;                    // rays for the next pass
    uint32_t *in_count;             // device counter written by the previous pass
    uint32_t *out_count;
    uint32_t *in_cursor;            // work-fetch cursor of this pass
    const uint32_t *in_perm;        // optional: coherence-sorted order of the first n_sorted input records (nullptr = as emitted)
    uint32_t n_sorted;              // records beyond it (the pass grew past the host's estimate) are read in emission order
    const uint32_t *ring_start;     // optional (sorted, heavy-first passes): first sorted index of cost ring 1, 2, 3 at [1..3];
                                    // warps take fewer rays per fetch from the expensive rings (kernels.cuh)
    uint32_t fetch_sizes;           // rays per fetch from rings 0, 1, 2 (one byte each; ring 3 and unsorted passes: 32)
    uint32_t capacity;              // in records
    uint32_t rec4;                  // record size in float4 units
};

struct ControlDev {
    uint32_t *tile_cursor;          // atomic block queue of the primary pass
    volatile int *abort_flag;       // host-mapped; renderer::state == CANCEL (reference src/render.cpp:333,412)
    unsigned long long *counters;   // ntr_counters layout (8 x u64)
    uint32_t *overflow;             // set when a wavefront queue was too small
    unsigned long long *fetch_stats;  // diagnostic builds (-DNTR_FETCH_STATS=1): [0] longest fetch, [1] sum, [2] fetches, [8+k] fetches of 2^k..2^(k+1) cycles
};
