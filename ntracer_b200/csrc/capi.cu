// capi.cu -- host side of the backend: C ABI of include/ntracer_b200.h, device arena builder
// ("geom_allocator" in the north-star sense), stream / event / wavefront-queue management.
// There is no CPU rendering path in this file or anywhere else in the library.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <new>
#include <string>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "arena_pack.h"
#include "errors.h"
#include "kernels.cuh"

using namespace ntr;

namespace {

thread_local std::string g_err;

void set_error(const char *fmt, va_list ap) {
    char buf[512];
    vsnprintf(buf, sizeof buf, fmt, ap);
    g_err = buf;
}

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    set_error(fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return fail(e_ == cudaErrorMemoryAllocation ? NTR_ERR_MEMORY : NTR_ERR_RUNTIME, "%s failed: %s", #expr, \
                        cudaGetErrorString(e_));                                                         \
    } while (0)

constexpr int kMaxPasses = 64;          // upper bound on max_reflect_depth handled by the control block

// control block layout (uint32 words); an adaptively supersampled frame runs a second round of passes with queue
// counters and cursors of its own (CTL_COUNT0B / CTL_CURSOR0B), the halo and refine passes' cursors and the number of
// refined pixels (written by the device, read by the refine pass and the host)
constexpr int kSlabMax = 4;
constexpr int kSchedViews = kSlabMax, kSchedSlots = kSlabMax + 1;     // tile schedules: one per control slot, one for views calls
enum { CTL_TILE_CURSOR = 0, CTL_OVERFLOW = 1, CTL_COUNT0 = 2, CTL_CURSOR0 = CTL_COUNT0 + kMaxPasses + 1,
       CTL_COUNT0B = CTL_CURSOR0 + kMaxPasses + 1, CTL_CURSOR0B = CTL_COUNT0B + kMaxPasses + 1,
       CTL_HALO_CURSOR = CTL_CURSOR0B + kMaxPasses + 1, CTL_LIST_CURSOR, CTL_REFINED, CTL_WORDS };

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__global__ void pack_kernel(const __grid_constant__ FrameDev f);
__global__ void classify_kernel(const __grid_constant__ FrameDev f, float threshold, unsigned char *mask);
__global__ void ray_keys_kernel(const float4 *recs, uint32_t rec4, uint32_t n, const uint32_t *count, uint32_t capacity, int D,
                                const __grid_constant__ SceneDev s, uint32_t *keys, uint32_t *idx, int heavy_first);
__global__ void ring_bounds_kernel(const uint32_t *sorted_keys, uint32_t n, const uint32_t *count, uint32_t capacity, uint32_t *ring_start);

}  // namespace

// One open frame of the begin/end interface: its own device frame, a pinned staging buffer for pageable destinations
// and the event that marks the end of its device->host copy.
struct FrameSlot {
    unsigned char *d_buf = nullptr; size_t d_cap = 0;
    unsigned char *h_stage = nullptr; size_t h_cap = 0;
    unsigned char *d_aov = nullptr; size_t d_aov_cap = 0;          // AOVs of a views launch (device) and their pinned staging
    unsigned char *h_aov = nullptr; size_t h_aov_cap = 0;
    cudaEvent_t rendered = nullptr, copied = nullptr;
    unsigned char *dst = nullptr;
    size_t pitch = 0, row_bytes = 0;
    int height = 0;
    bool open = false, staged = false;
    uint64_t ticket = 0;
};

int ntr_fail(int code, const char *fmt, ...) {        // errors.h: for builder.cpp
    va_list ap;
    va_start(ap, fmt);
    set_error(fmt, ap);
    va_end(ap);
    return code;
}

struct ntr_scene {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing_valid = false;
    SceneDev dev{};
    CameraDev cam{};
    void *arena = nullptr;
    size_t arena_bytes = 0;
    float *d_lights = nullptr;
    int base_flags = 0;
    bool any_reflective = false;
    bool instrumented = false;
    int tree_depth = 0;
    uint32_t *d_ctl = nullptr;
    unsigned long long *d_counters = nullptr;
    // abort words (mapped pinned): [0] = the synchronous entry points and asynchronous ntr_render_device frames,
    // [1 + k] = frame slot k of ntr_render_begin / ntr_render_end.  One word per open frame: an abort hits exactly
    // the frames that were open when it came, and a frame begun afterwards starts clean.
    int *h_abort = nullptr;
    int *d_abort = nullptr;
    int abort_idx = 0;                  // word the frame being enqueued polls
    float *d_accum = nullptr; size_t accum_cap = 0;
    unsigned char *d_packed = nullptr; size_t packed_cap = 0;
    int32_t *d_ids = nullptr; float *d_dists = nullptr; size_t ids_cap = 0;
    float4 *d_queue[2] = {nullptr, nullptr};
    uint32_t queue_capacity = 0;
    void *d_scratch = nullptr; size_t scratch_cap = 0;
    // cost-sorted tile schedule, one per control slot (valid for one window / interleave geometry at a time).  The slabs of
    // a frame run side by side on their own streams, so each needs its own: slot k's order is written by the
    // order_tiles_kernel behind slot k's primary pass, and slot k is reused only on the same stream or after its frame_done.
    // Views calls (ntr_render_views) keep one more schedule of their own, at kSchedViews.
    unsigned long long *d_tile_cost[kSchedSlots] = {};
    uint32_t *d_tile_order[kSchedSlots] = {};
    size_t tile_cap[kSchedSlots] = {};
    long long sched_key[kSchedSlots] = {-1, -1, -1, -1, -1};      // geometry the stored order belongs to
    bool sched_ready[kSchedSlots] = {};                            // an order has been computed for sched_key
    // coherence sort of the wavefront queues (keys, permutation, CUB scratch)
    uint32_t *d_keys[2] = {nullptr, nullptr}, *d_perm[2] = {nullptr, nullptr};
    void *d_sort_tmp = nullptr; size_t sort_tmp_bytes = 0; uint32_t sort_cap = 0;
    bool sort_rays = true;
    // ntr_render of single-pass frames into pinned memory: the frame is cut into slabs of tile rows, one persistent
    // kernel + copy per slab on its own stream, so that all but the last slab cross PCIe underneath the tracing
    int ctl_slot = 0;
    // the last frame enqueued with each control block: a frame on ANOTHER stream waits for it before it resets the block
    // (asynchronous ntr_render_device frames return while their persistent kernel still runs)
    cudaEvent_t frame_done[kSlabMax] = {};
    cudaStream_t frame_stream[kSlabMax] = {};
    cudaStream_t slab_stream[kSlabMax] = {};
    cudaEvent_t slab_done[kSlabMax] = {};
    bool slabs = true;                  // NTR_NO_SLABS=1 switches it off
    // bounce passes of scenes with big leaves start the rays nearest the scene centre first (ray_keys_kernel) and hand
    // them out a few per warp (fetch_sizes below); NTR_HEAVY_FIRST / NTR_ADAPTIVE_FETCH = 0|1 override
    bool heavy_first = false, adaptive_fetch = false;
    uint32_t max_leaf = 0;              // items in the largest leaf of the tree
    uint32_t *d_ring = nullptr;
    uint32_t fetch_sizes = 4u | (8u << 8) | (16u << 16);      // NTR_FETCH_SIZES=a,b,c: rays per fetch from cost rings 0, 1, 2
    bool no_tile_sched = false;         // NTR_TILE_SCHED=0: row-major tile order always
    bool force_tile_sched = false;      // NTR_TILE_SCHED=1: cost-sorted tile hand-out on whole frames too (heavy-tailed scenes, DESIGN section 8)
    bool zero_copy = false;             // NTR_ZEROCOPY=1: ntr_render stores single-pass frames straight into pinned destinations
    uint32_t queue_init = 0;            // NTR_QUEUE_INIT: initial queue capacity override (tests force the regrow path)
    float pass_ns_per_ray = 0.0f;       // measured cost of the wavefront passes of the previous frame (0 = unknown)
    uint32_t prev_pass_count[kMaxPasses + 2] = {};      // rays per pass of the previous frame: the sort sizes of this one
    // diagnostic per-pass timing (NTR_PASS_TIMING=1): events between the passes of one frame
    cudaEvent_t pass_ev[kMaxPasses + 4] = {};
    int n_pass_ev = 0;
    bool pass_timing = false;
    ntr_counters counters{};
    int ss = 1;                         // supersampling factor (ntr_scene_set_supersampling), read when a frame is enqueued
    float ss_threshold = -1.0f;         // adaptive supersampling threshold (ntr_scene_set_supersampling_threshold), < 0: off
    // adaptive frames: refine mask of the launch's own pixels, the compacted list of refined slots, CUB scratch, and the
    // pass sizes of the refine round in the previous frame (its sort sizes)
    unsigned char *d_mask = nullptr; size_t mask_cap = 0;
    uint32_t *d_list = nullptr; size_t list_cap = 0;
    void *d_select_tmp = nullptr; size_t select_tmp_cap = 0;
    uint32_t prev_pass_count2[kMaxPasses + 2] = {};
    // what ntr_last_refine_mask reports: the geometry of the last frame, whether it was adaptive, its halo and refined pixels
    struct {
        bool valid = false, adaptive = false;
        int win_w = 0, win_h = 0, out_rows = 0, trf = 0, trs = 1, compact = 0;
        uint64_t halo = 0, refined = 0;
    } last;
    // pageable destinations (what BlockingRenderer.render is handed: a bytearray): frames cross PCIe into this pinned
    // staging buffer in row chunks, and the host copies chunk k into the caller's buffer while chunk k+1 is in flight
    unsigned char *h_stage = nullptr; size_t h_stage_cap = 0;
    cudaEvent_t stage_ev[8] = {};
    uint32_t *h_ctl = nullptr;              // pinned read-back of the control block and the counters (frame_readback)
    unsigned long long *h_cnt = nullptr;
    uint64_t launches = 0;
    int grid_blocks[512] = {};         // per variant flags (NTR_F_SS, NTR_F_LIST, NTR_F_VIEWS, NTR_F_AOV and NTR_F_PROJ included)
    // NTR_F_WIDE builds (96 registers, 5 CTAs per SM): for frames sharded over 4 or more GPUs, whose passes all end in a few
    // long rays (measured, config 4: 1/4 share 20.9 -> 19.9 ms, 1/8 share 15.2 -> 14.4 ms; 1/2 share and whole frames lose
    // 2..12 %).  Picking the build per pass from pass times measured on the second and third frame of a view gained another
    // 0.7 % on whole frames when it measured right and lost 4 % when one noisy sample misled it (calls 27, 28): not kept.
    // NTR_WIDE=0|1: never | always.
    int wide_mode = -1;
    int warp_path = 0;                  // 1: bounce passes use the warp-synchronous kernels (scenes with big leaves), 2: every pass; NTR_WARP overrides
    const KernelSet *(*kset)(int) = nullptr;
    std::atomic<bool> busy{false};
    // batches of views (ntr_render_views): the cameras of the call on the device, and the wavefront statistics of views calls.
    // They are kept apart from the single frames' (pass_ns_per_ray, prev_pass_count) -- as the tile schedule is (kSchedViews)
    // -- so that a frame rendered after a views call makes the decisions it would have made without it, and vice versa.
    CameraDev *d_views = nullptr; size_t views_cap = 0;
    float views_pass_ns_per_ray = 0.0f;
    uint32_t views_prev_pass_count[kMaxPasses + 2] = {};
    uint32_t views_per_launch = 0;      // NTR_VIEWS_PER_LAUNCH: views per launch of a views call (0: from kViewsSampleCap)
    // batches of caller-given rays (ntr_render_rays): wavefront statistics of their own, kept apart like the views calls'; the
    // grid of the ray-fed primary pass per build (FLAGS & 3); NTR_RAYS_PER_LAUNCH: rays per launch (0: kRaysPerLaunch)
    float rays_pass_ns_per_ray = 0.0f;
    uint32_t rays_prev_pass_count[kMaxPasses + 2] = {};
    int rays_grid[4] = {};
    uint32_t rays_per_launch = 0;
    // the projection (ntr_scene_set_projection), read when a frame is enqueued, and the wavefront statistics of projected frames,
    // kept apart like the views calls' (projected frames keep no tile schedule), so that a perspective frame makes the decisions
    // it would have made without them
    int proj = NTR_PROJ_PERSPECTIVE;
    float proj_param = 0.0f;
    float proj_pass_ns_per_ray = 0.0f;
    uint32_t proj_prev_pass_count[kMaxPasses + 2] = {}, proj_prev_pass_count2[kMaxPasses + 2] = {};
    // begin/end frames (ntr_render_begin / ntr_render_end); a views call uses their device buffers, staging buffers, events and
    // copy stream for its double-buffered launches
    FrameSlot slots[NTR_FRAMES_IN_FLIGHT];
    cudaStream_t copy_stream = nullptr;
    uint64_t next_ticket = 0;
};

namespace {

const KernelSet *(*kernel_family(int dim))(int) {
    switch (dim) {
        case 3: return &kernel_set_d3;
        case 4: return &kernel_set_d4;
        case 5: return &kernel_set_d5;
        case 6: return &kernel_set_d6;
        case 7: return &kernel_set_d7;
        case 8: return &kernel_set_d8;
        case 9: return &kernel_set_d9;
        case 10: return &kernel_set_d10;
        default: return &kernel_set_dn;     // run-time dimension kernels (the reference's generic tracern)
    }
}

int validate_desc(const ntr_scene_desc *d, int *tree_depth_out) {
    if (!d) return fail(NTR_ERR_VALUE, "scene description is NULL");
    if (d->dim < 3 || d->dim > NTR_MAX_DIM) return fail(NTR_ERR_VALUE, "dimension must be between 3 and %d", NTR_MAX_DIM);
    if (d->kind != NTR_SCENE_BOX && d->kind != NTR_SCENE_COMPOSITE) return fail(NTR_ERR_VALUE, "unknown scene kind %d", d->kind);
    *tree_depth_out = 0;
    if (d->kind == NTR_SCENE_BOX) return NTR_OK;
    if (d->batch_size < 1 || d->batch_size > 64) return fail(NTR_ERR_VALUE, "batch_size must be in 1..64");
    if (!d->boundary) return fail(NTR_ERR_VALUE, "composite scene needs a boundary");
    if (d->bg_gradient_axis < 0 || d->bg_gradient_axis >= d->dim) return fail(NTR_ERR_VALUE, "bg_gradient_axis out of range");
    if (d->max_reflect_depth < 0 || d->max_reflect_depth > kMaxPasses - 1)
        return fail(NTR_ERR_VALUE, "max_reflect_depth must be between 0 and %d (one wavefront pass per depth)", kMaxPasses - 1);
    if (d->n_nodes && !d->nodes) return fail(NTR_ERR_VALUE, "nodes is NULL");
    if (d->n_leaf_refs && !d->leaf_refs) return fail(NTR_ERR_VALUE, "leaf_refs is NULL");
    if (d->n_simplex && (!d->simplex || !d->simplex_mat)) return fail(NTR_ERR_VALUE, "simplex / simplex_mat is NULL");
    if (d->n_solids && (!d->solids || !d->solid_mat)) return fail(NTR_ERR_VALUE, "solids / solid_mat is NULL");
    if (d->n_materials && !d->materials) return fail(NTR_ERR_VALUE, "materials is NULL");
    if ((d->n_point_lights && !d->point_lights) || (d->n_global_lights && !d->global_lights)) return fail(NTR_ERR_VALUE, "lights array is NULL");
    if (d->root != NTR_NULL_NODE && d->root >= d->n_nodes) return fail(NTR_ERR_VALUE, "root node out of range");
    if (d->n_materials == 0 && (d->n_simplex || d->n_solids)) return fail(NTR_ERR_VALUE, "primitives without materials");
    for (uint32_t i = 0; i < d->n_simplex; ++i)
        if (d->simplex_mat[i] < 0 || (uint32_t)d->simplex_mat[i] >= d->n_materials)
            return fail(NTR_ERR_VALUE, "simplex %u: material index out of range", i);
    for (uint32_t i = 0; i < d->n_solids; ++i) {
        if (d->solid_mat[i] < 0 || (uint32_t)d->solid_mat[i] >= d->n_materials)
            return fail(NTR_ERR_VALUE, "solid %u: material index out of range", i);
        const int type = (int)d->solids[(size_t)i * (1 + 2 * d->dim * d->dim + d->dim)];
        if (type != NTR_SOLID_CUBE && type != NTR_SOLID_SPHERE) return fail(NTR_ERR_VALUE, "solid %u: unknown type", i);
    }
    for (uint32_t i = 0; i < d->n_nodes; ++i) {
        const ntr_node &n = d->nodes[i];
        if (n.meta & NTR_LEAF_FLAG) {
            if ((uint64_t)n.w1 + n.w2 > d->n_leaf_refs) return fail(NTR_ERR_VALUE, "leaf %u: item range out of bounds", i);
            for (uint32_t k = 0; k < n.w2; ++k) {
                const uint32_t r = d->leaf_refs[n.w1 + k], kind = r >> 30, idx = r & NTR_IDX_MASK;
                if (kind == NTR_REF_SIMPLEX) { if (idx >= d->n_simplex) return fail(NTR_ERR_VALUE, "leaf %u: simplex index out of range", i); }
                else if (kind == NTR_REF_BATCH) {
                    if ((uint64_t)idx + d->batch_size > d->n_simplex) return fail(NTR_ERR_VALUE, "leaf %u: batch out of range", i);
                    if (d->batch_size % 4) return fail(NTR_ERR_VALUE, "batch items need a batch_size that is a multiple of 4");
                }
                else if (kind == NTR_REF_SOLID) { if (idx >= d->n_solids) return fail(NTR_ERR_VALUE, "leaf %u: solid index out of range", i); }
                else return fail(NTR_ERR_VALUE, "leaf %u: bad item type", i);
            }
        } else {
            if (n.meta >= (uint32_t)d->dim) return fail(NTR_ERR_VALUE, "branch %u: axis out of range", i);
            if ((n.w2 != NTR_NULL_NODE && n.w2 >= d->n_nodes) || (n.w3 != NTR_NULL_NODE && n.w3 >= d->n_nodes))
                return fail(NTR_ERR_VALUE, "branch %u: child out of range", i);
        }
    }
    // depth (also rejects cycles: a path longer than the stack the kernels carry is an error either way)
    int depth = 0;
    if (d->root != NTR_NULL_NODE) {
        std::vector<std::pair<uint32_t, int>> st;
        st.push_back({d->root, 1});
        size_t visited = 0;
        while (!st.empty()) {
            auto [n, dep] = st.back();
            st.pop_back();
            if (++visited > (size_t)d->n_nodes * 2 + 2) return fail(NTR_ERR_VALUE, "k-d tree is not a tree");
            if (dep > NTR_MAX_TREE_DEPTH) return fail(NTR_ERR_VALUE, "k-d tree deeper than %d", NTR_MAX_TREE_DEPTH);
            depth = std::max(depth, dep);
            const ntr_node &nd = d->nodes[n];
            if (nd.meta & NTR_LEAF_FLAG) continue;
            if (nd.w2 != NTR_NULL_NODE) st.push_back({nd.w2, dep + 1});
            if (nd.w3 != NTR_NULL_NODE) st.push_back({nd.w3, dep + 1});
        }
    }
    *tree_depth_out = depth;
    return NTR_OK;
}

void fill_params(SceneDev &dev, const ntr_scene_desc *d) { fill_scene_params(dev, d, kMaxPasses - 1); }

int upload_lights(ntr_scene *sc, const ntr_scene_desc *d) {
    const size_t stride = d->dim + 3;
    const size_t n = ((size_t)d->n_point_lights + d->n_global_lights) * stride;
    if (sc->d_lights) { cudaFree(sc->d_lights); sc->d_lights = nullptr; }
    sc->dev.n_point = (int)d->n_point_lights;
    sc->dev.n_global = (int)d->n_global_lights;
    sc->dev.point_lights = sc->dev.global_lights = nullptr;
    if (!n) return NTR_OK;
    std::vector<float> h(n);
    if (d->n_point_lights) memcpy(h.data(), d->point_lights, sizeof(float) * d->n_point_lights * stride);
    if (d->n_global_lights) memcpy(h.data() + d->n_point_lights * stride, d->global_lights, sizeof(float) * d->n_global_lights * stride);
    CUDA_TRY(cudaMalloc(&sc->d_lights, n * sizeof(float)));
    CUDA_TRY(cudaMemcpy(sc->d_lights, h.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    sc->dev.point_lights = sc->d_lights;
    sc->dev.global_lights = sc->d_lights + d->n_point_lights * stride;
    return NTR_OK;
}

// Builds the single device arena: nodes | leaf refs | simplex records | solid records | materials.
int build_arena(ntr_scene *sc, const ntr_scene_desc *d) {
    std::vector<unsigned char> h;
    ArenaLayout L;
    try { pack_arena(d, h, L); } catch (const std::bad_alloc &) { return fail(NTR_ERR_MEMORY, "out of host memory building the arena"); }
    CUDA_TRY(cudaMalloc(&sc->arena, L.total));
    sc->arena_bytes = L.total;
    CUDA_TRY(cudaMemcpy(sc->arena, h.data(), L.total, cudaMemcpyHostToDevice));
    bind_arena(sc->dev, d, L, static_cast<const unsigned char *>(sc->arena));
    sc->any_reflective = L.any_reflective;
    sc->base_flags = (L.any_transparent || d->n_solids) ? NTR_F_GENERAL : 0;
    return NTR_OK;
}

int ensure(void **p, size_t *cap, size_t need) {
    if (*cap >= need && *p) return NTR_OK;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    const size_t n = align_up(need + need / 8, 256);
    CUDA_TRY(cudaMalloc(p, n));
    *cap = n;
    return NTR_OK;
}

int ensure_queues(ntr_scene *sc, uint32_t capacity) {
    if (sc->queue_capacity >= capacity && sc->d_queue[0]) return NTR_OK;
    for (int i = 0; i < 2; ++i) if (sc->d_queue[i]) { cudaFree(sc->d_queue[i]); sc->d_queue[i] = nullptr; }
    sc->queue_capacity = 0;
    const uint32_t rec4 = 2 + 2 * ((sc->dev.dim + 3) / 4);
    for (int i = 0; i < 2; ++i) CUDA_TRY(cudaMalloc(&sc->d_queue[i], (size_t)capacity * rec4 * sizeof(float4)));
    sc->queue_capacity = capacity;
    return NTR_OK;
}

int grid_for(ntr_scene *sc, int flags) {
    if (!sc->grid_blocks[flags]) {
        int per_sm = sc->kset(flags)->max_blocks_per_sm();
        if (per_sm < 1) per_sm = 1;
        sc->grid_blocks[flags] = per_sm * sc->sm_count;      // persistent: a whole number of CTAs per SM
    }
    return sc->grid_blocks[flags];
}

void fill_format(FormatDev &o, const ntr_image_format *f) {
    memset(&o, 0, sizeof o);
    o.n_channels = f->n_channels; o.bytes_per_pixel = f->bytes_per_pixel; o.reversed = f->reversed; o.pitch = f->pitch;
    for (int i = 0; i < f->n_channels; ++i) {
        o.f_r[i] = f->channels[i].f_r; o.f_g[i] = f->channels[i].f_g; o.f_b[i] = f->channels[i].f_b; o.f_c[i] = f->channels[i].f_c;
        o.bits[i] = f->channels[i].bit_size; o.tfloat[i] = f->channels[i].tfloat;
    }
}

int check_format(const ntr_image_format *f) {
    if (!f) return fail(NTR_ERR_VALUE, "image format is NULL");
    if (f->width < 1 || f->height < 1) return fail(NTR_ERR_VALUE, "width and height must be at least 1");
    if (f->n_channels < 0 || f->n_channels > NTR_MAX_CHANNELS) return fail(NTR_ERR_VALUE, "too many channels");
    int bits = 0;
    for (int i = 0; i < f->n_channels; ++i) {
        const ntr_channel &c = f->channels[i];
        if (c.tfloat) { if (c.bit_size != 32) return fail(NTR_ERR_VALUE, "if \"tfloat\" is true, \"bit_size\" can only be 32"); }
        else if (c.bit_size > 31) return fail(NTR_ERR_VALUE, "\"bit_size\" cannot be greater than 31 (unless \"tfloat\" is true)");
        else if (c.bit_size < 1) return fail(NTR_ERR_VALUE, "\"bit_size\" cannot be less than 1");
        bits += c.bit_size;
    }
    if (bits > 128) return fail(NTR_ERR_VALUE, "Too many bytes per pixel. The maximum is 16.");
    if (f->bytes_per_pixel != (bits + 7) / 8) return fail(NTR_ERR_VALUE, "bytes_per_pixel does not match the channels");
    if (f->pitch < f->width * f->bytes_per_pixel)
        return fail(NTR_ERR_VALUE, "invalid image format: \"pitch\" must be at least \"width\" times the pixel size in bytes");
    return NTR_OK;
}

// The AOVs of a batch of views (ntr_aov_buffers): p[k] is where kind k of view 0 goes (nullptr: not wanted), kind k taking
// aov_bytes(k, dim) bytes per pixel -- 0 ids (int32), 1 depth (float), 2 normals (dim floats)
struct AovTarget {
    void *p[3] = {nullptr, nullptr, nullptr};
    bool any() const { return p[0] || p[1] || p[2]; }
};
static size_t aov_bytes(int k, int dim) { return k == 2 ? 4 * (size_t)dim : 4; }
// bytes per pixel of the AOVs wanted
static size_t aov_pixel_bytes(const AovTarget &a, int dim) {
    size_t b = 0;
    for (int k = 0; k < 3; ++k) if (a.p[k]) b += aov_bytes(k, dim);
    return b;
}
// a's arrays from pixel `pix` on
static AovTarget aov_offset(const AovTarget &a, size_t pix, int dim) {
    AovTarget o;
    for (int k = 0; k < 3; ++k) if (a.p[k]) o.p[k] = static_cast<unsigned char *>(a.p[k]) + pix * aov_bytes(k, dim);
    return o;
}
// the arrays of `want` for npix pixels laid out one after the other in buf
static AovTarget aov_packed(unsigned char *buf, const AovTarget &want, size_t npix, int dim) {
    AovTarget o;
    for (int k = 0; k < 3; ++k) if (want.p[k]) { o.p[k] = buf; buf += npix * aov_bytes(k, dim); }
    return o;
}

struct RenderTarget {
    int out_mode;               // what the caller wants
    unsigned char *packed = nullptr;
    float *accum = nullptr;
    int32_t *ids = nullptr;
    float *dists = nullptr;
    AovTarget aov;              // a batch of views or rays only: its AOVs (device memory)
    const float *ray_o = nullptr, *ray_d = nullptr;     // NTR_OUT_RAYS: the rays (device memory, n x D), n = the window width
};

// Supersampling factor of a frame: the hit-id hook and a batch of rays trace one ray per pixel whatever the scene's factor
int frame_ss(const ntr_scene *sc, int out_mode) { return out_mode == NTR_OUT_IDS || out_mode == NTR_OUT_RAYS ? 1 : sc->ss; }
// Adaptive supersampling: a factor above 1 and a threshold.  Such frames always take the accumulator route
bool frame_adaptive(const ntr_scene *sc, int out_mode) { return frame_ss(sc, out_mode) > 1 && sc->ss_threshold >= 0.0f; }

// Pixels of the halo of frame f that are traced (trace_core.cuh: halo_pixel): the column right of the window and, per owned
// tile row, the row below it (every pixel but the one past the window is valid or not alike)
uint64_t count_halo(const FrameDev &f) {
    uint64_t n = 0;
    int wx = 0, wy = 0;
    for (int r = 0; r < f.out_rows; ++r) n += halo_pixel(f, (uint32_t)r, &wx, &wy);
    for (int k = 0; k < owned_tile_rows(f); ++k) {
        const uint32_t h = (uint32_t)f.out_rows + (uint32_t)k * (uint32_t)(f.win_w + 1);
        n += (uint64_t)halo_pixel(f, h, &wx, &wy) * (uint64_t)f.win_w + halo_pixel(f, h + (uint32_t)f.win_w, &wx, &wy);
    }
    return n;
}

// Enqueues every kernel of one frame on `st`.  view = (width,height), window = (x0,y0,w,h).
// A supersampled frame (factor ss > 1) traces the ss-times-larger view: FrameDev describes that view, while the window,
// the tile grid and every output stay in output pixels (slabs, tile-row interleaving, compact strips and the 1x1 window of
// ntr_calculate_color work unchanged).
// An adaptively supersampled frame (frame_adaptive) runs in two rounds: the plain frame -- the base primary pass into the
// accumulator, the halo pass (list-driven, factor 1) and the bounce passes -- then classify_kernel marks the pixels to
// refine and compacts them into a list, the list-driven pass traces them at factor ss over their accumulator slots, the
// second round of bounce passes follows, and pack_kernel packs the frame.
// A batch of views (n_views > 0, whole frames at a factor >= 1, never adaptive) runs the NTR_F_VIEWS primary pass over the
// cameras views[0 .. n_views): view v has accumulator slots v * npix .. and its packed frame at tgt.packed + v * pitch * win_h;
// the bounce passes and pack_kernel are the single frame's, over all views at once.
// A batch of caller-given rays (tgt.out_mode NTR_OUT_RAYS, factor 1) is a win_w x 1 window: render_rays_kernel traces ray i into
// accumulator slot i, the bounce passes are the single frame's, nothing is packed, no tile schedule is kept and the refine-mask
// record is left alone.
// Under a projection other than the perspective one (sc->proj) every primary pass runs an NTR_F_PROJ build: a batch of views
// its views builds; a single frame the views build too, as one view (FrameDev::n_views = 1, views = nullptr: the kernel's
// camera) -- a hit-id frame with its ids and depth stored as AOVs -- and the list passes of an adaptive frame the NTR_F_LIST
// one.  Such frames keep no tile schedule and keep wavefront statistics of their own.
int enqueue_frame(ntr_scene *sc, cudaStream_t st, int width, int height, int x0, int y0, int win_w, int win_h,
                  const ntr_image_format *fmt, const RenderTarget &tgt, int tile_row_first, int tile_row_step,
                  int compact, bool *used_passes, const CameraDev *views = nullptr, uint32_t n_views = 0) {
    uint32_t *const d_ctl = sc->d_ctl + (size_t)sc->ctl_slot * CTL_WORDS;                 // one control block per slab
    unsigned long long *const d_counters = sc->d_counters + (size_t)sc->ctl_slot * 8;
    if (sc->frame_done[sc->ctl_slot] && sc->frame_stream[sc->ctl_slot] != st)
        CUDA_TRY(cudaStreamWaitEvent(st, sc->frame_done[sc->ctl_slot], 0));
    FrameDev f;
    memset(&f, 0, sizeof f);
    const bool adaptive = frame_adaptive(sc, tgt.out_mode);
    const int ss = adaptive ? 1 : frame_ss(sc, tgt.out_mode);          // the base of an adaptive frame is the plain frame
    f.ss = ss;
    f.width = width * ss; f.height = height * ss;
    // flat_origin_ray_source::set_params (tracer.hpp:65-69)
    f.half_w = (float)f.width / 2.0f;
    f.half_h = (float)f.height / 2.0f;
    f.fovI = tanf(sc->dev.fov / 2) / f.half_w;
    f.x0 = x0; f.y0 = y0; f.win_w = win_w; f.win_h = win_h;
    f.tiles_x = (win_w + NTR_TILE - 1) / NTR_TILE;
    f.tiles_y = (win_h + NTR_TILE - 1) / NTR_TILE;
    f.tile_row_first = tile_row_first; f.tile_row_step = tile_row_step < 1 ? 1 : tile_row_step; f.compact = compact;
    if (fmt) fill_format(f.fmt, fmt);
    f.views = views; f.n_views = n_views;
    const bool rays = tgt.out_mode == NTR_OUT_RAYS;
    const bool proj = !rays && sc->proj != NTR_PROJ_PERSPECTIVE;
    AovTarget aovs = tgt.aov;
    if (proj && tgt.out_mode == NTR_OUT_IDS) { aovs.p[0] = tgt.ids; aovs.p[1] = tgt.dists; }
    const bool aov = (n_views || rays || proj) && aovs.any();
    if (proj) {
        f.proj = sc->proj;
        f.proj_k = projection_k(sc->proj, sc->proj_param, f.half_w);
        if (!n_views) f.n_views = 1;
    }
    if (aov) {
        f.aov_ids = static_cast<int32_t *>(aovs.p[0]);
        f.aov_depth = static_cast<float *>(aovs.p[1]);
        f.aov_normals = static_cast<float *>(aovs.p[2]);
        // the plain frame's ray parameters, as ntr_primary_hit_ids sets them (factor 1)
        f.aov_half_w = (float)width / 2.0f;
        f.aov_half_h = (float)height / 2.0f;
        f.aov_fovI = tanf(sc->dev.fov / 2) / f.aov_half_w;
        if (proj) f.aov_proj_k = projection_k(sc->proj, sc->proj_param, f.aov_half_w);
    }
    const size_t nv = n_views ? n_views : 1;
    // wavefront statistics of the previous frame (of the previous views call, for a batch of views)
    float &pass_ns_per_ray = rays ? sc->rays_pass_ns_per_ray : n_views ? sc->views_pass_ns_per_ray
                             : proj ? sc->proj_pass_ns_per_ray : sc->pass_ns_per_ray;

    // Scenes with big leaves: the bounce passes run the warp-synchronous kernels (incoherent rays; lanes that run out of
    // work help the ones parked at big leaves), the primary pass every lane for itself (the 32 rays of an 8x4 pixel block
    // walk the same leaves: nothing to share out, and the per-lane form is the leaner code).  Measured, config 4 per
    // pass (ms): per-lane 11.4 12.5 7.3 10.8 10.5 | warp 13.8 11.6 6.8 9.2 7.7.  NTR_WARP=0|1|2: never | bounces | all passes.
    int flags = sc->base_flags | (sc->instrumented ? NTR_F_COUNT : 0);
    const int primary_flags = flags | (sc->warp_path == 2 ? NTR_F_WARP : 0);
    const int bounce_flags = flags | (sc->warp_path ? NTR_F_WARP : 0);
    const bool composite = sc->dev.kind == NTR_SCENE_COMPOSITE;
    const bool passes = composite && tgt.out_mode != NTR_OUT_IDS && sc->any_reflective && sc->dev.max_depth > 0;
    *used_passes = passes;

    {
        const int my_rows = f.tile_row_first < f.tiles_y ? (f.tiles_y - f.tile_row_first + f.tile_row_step - 1) / f.tile_row_step : 0;
        f.out_rows = compact ? my_rows * NTR_TILE : win_h;
    }
    const size_t npix = (size_t)win_w * f.out_rows;
    const size_t nhalo = adaptive ? halo_slots(f) : 0;          // accumulator slots behind the window's own pixels
    f.packed = tgt.packed; f.accum = tgt.accum; f.ids = tgt.ids; f.dists = tgt.dists;
    f.out_mode = tgt.out_mode;
    if (adaptive || (passes && tgt.out_mode == NTR_OUT_PACKED)) {
        int rc = ensure((void **)&sc->d_accum, &sc->accum_cap, (npix * nv + nhalo) * 3 * sizeof(float));
        if (rc) return rc;
        f.accum = sc->d_accum;
        f.out_mode = NTR_OUT_ACCUM;
    }
    if (passes) {
        // each pass can emit at most (1 + transparent layers) rays per input ray; start with 2 rays per traced sample
        // (ss*ss per pixel; capped at 2^26 records -- 4 GB per queue in 4 dimensions -- unless a plain frame needs more)
        // and let the overflow check regrow (ntr_counters.queue_overflows)
        const uint64_t plain = (uint64_t)(npix * nv + nhalo) * 2;
        const uint64_t want = sc->queue_init ? sc->queue_init
                                             : std::max<uint64_t>(std::min<uint64_t>(plain * ss * ss, std::max<uint64_t>(plain, 1ull << 26)), 1u << 16);
        if (sc->queue_capacity < want) {
            int rc = ensure_queues(sc, (uint32_t)std::min<uint64_t>(want, 0x7FFFFFFFu));
            if (rc) return rc;
        }
    }

    // ---- tile schedule: reuse the order measured on the previous frame of the same geometry ----
    const size_t n_tiles = (size_t)(f.out_rows ? (compact ? f.out_rows / NTR_TILE : (f.tiles_y - tile_row_first + f.tile_row_step - 1) / f.tile_row_step) : 0) * f.tiles_x;
    const long long key = (((((long long)win_w * 65536 + win_h) * 64 + tile_row_first) * 64 + f.tile_row_step) * 4 + x0 % 2 * 2 + y0 % 2) * 8 + (ss - 1);
    // measured: the cost-sorted schedule pays when the frame is sharded over GPUs (8 GPUs, config 2: strip render
    // 0.258 -> 0.203 ms) -- each rank then has only ~2 blocks per warp and the tail matters -- but costs ~8 % on a
    // whole frame on one GPU (loss of row-major locality + the cost bookkeeping), so it is used for sharded renders --
    // and for whole frames of scenes with giant leaves, whose few blocks through the centre cost 10-90x the mean
    // (config 4: primary pass 11.2-11.6 -> 10.4 ms, frame 43.3 -> 42.4 ms, calls 17 and 20)
    const bool use_sched = n_tiles >= 64 && composite && tgt.out_mode != NTR_OUT_IDS && !rays && !proj && !sc->no_tile_sched &&
                           (f.tile_row_step > 1 || sc->force_tile_sched || sc->max_leaf >= 256);
    const int slot = n_views ? kSchedViews : sc->ctl_slot;
    if (use_sched) {
        if (sc->tile_cap[slot] < n_tiles) {
            cudaFree(sc->d_tile_cost[slot]); cudaFree(sc->d_tile_order[slot]);
            sc->d_tile_cost[slot] = nullptr; sc->d_tile_order[slot] = nullptr; sc->tile_cap[slot] = 0;
            CUDA_TRY(cudaMalloc(&sc->d_tile_cost[slot], n_tiles * sizeof(unsigned long long)));
            CUDA_TRY(cudaMalloc(&sc->d_tile_order[slot], n_tiles * sizeof(uint32_t)));
            sc->tile_cap[slot] = n_tiles;
            sc->sched_key[slot] = -1;
        }
        if (sc->sched_key[slot] != key) {
            CUDA_TRY(cudaMemsetAsync(sc->d_tile_cost[slot], 0, n_tiles * sizeof(unsigned long long), st));
            sc->sched_key[slot] = key;
            sc->sched_ready[slot] = false;
        }
        f.tile_cost = sc->d_tile_cost[slot];
        f.tile_order = sc->sched_ready[slot] ? sc->d_tile_order[slot] : nullptr;
    }

    ControlDev ctl;
    ctl.tile_cursor = d_ctl + CTL_TILE_CURSOR;
    ctl.overflow = d_ctl + CTL_OVERFLOW;
    ctl.abort_flag = sc->d_abort + sc->abort_idx;
    ctl.counters = d_counters;
    ctl.fetch_stats = nullptr;
#if NTR_FETCH_STATS
    static unsigned long long *d_stats = nullptr;
    if (!d_stats) cudaMalloc(&d_stats, 80 * sizeof(unsigned long long));
    ctl.fetch_stats = d_stats;
    auto dump_stats = [&](const char *what, int depth) {
        unsigned long long h[80];
        cudaStreamSynchronize(st);
        cudaMemcpy(h, d_stats, sizeof h, cudaMemcpyDeviceToHost);
        cudaMemset(d_stats, 0, sizeof h);
        if (!h[2]) return;
        fprintf(stderr, "ntr fetch stats %s %d: fetches %llu, mean %.0f kcyc, longest %.0f kcyc; log2(cycles) histogram:", what, depth, h[2],
                (double)h[1] / h[2] / 1e3, (double)h[0] / 1e3);
        for (int k = 8; k < 40; ++k) if (h[8 + k]) fprintf(stderr, " %d:%llu", k, h[8 + k]);
        fprintf(stderr, "\n");
    };
    cudaMemsetAsync(d_stats, 0, 80 * sizeof(unsigned long long), st);
#endif
    CUDA_TRY(cudaMemsetAsync(d_ctl, 0, CTL_WORDS * sizeof(uint32_t), st));
    CUDA_TRY(cudaMemsetAsync(d_counters, 0, 8 * sizeof(unsigned long long), st));

    // passes that end in a few long rays (the late bounce passes of a frame, every pass of a share of a sharded frame)
    // run the 96-register build of scenes with giant leaves: see kernels.cuh, NTR_F_WIDE
    const bool wide_ok = sc->wide_mode != 0 && composite && passes && (flags & NTR_F_GENERAL) && sc->dev.dim <= 5 && sc->max_leaf >= 256;
    const uint32_t wide_now = wide_ok && (sc->wide_mode == 1 || f.tile_row_step >= 4) ? 0xFFFFFFFFu : 0u;
    auto wide_for = [&](int pass) { return (wide_now >> pass) & 1u ? (int)NTR_F_WIDE : 0; };
    // a supersampled primary pass runs the per-lane, non-wide NTR_F_SS build whatever NTR_WARP / NTR_WIDE say (kernels.cuh)
    // a batch of views, and any projected frame, runs the per-lane, non-wide NTR_F_VIEWS build at every factor, 1 included; no
    // more CTAs than the exact mailbox has columns
    const int pflags = n_views || proj ? (flags & (NTR_F_GENERAL | NTR_F_COUNT)) | NTR_F_VIEWS | (aov ? NTR_F_AOV : 0) | (proj ? NTR_F_PROJ : 0)
                       : ss > 1 ? (flags & (NTR_F_GENERAL | NTR_F_COUNT)) | NTR_F_SS : primary_flags | wide_for(0);
    const KernelSet *ks = sc->kset(pflags);
    int grid = grid_for(sc, pflags);
    if ((n_views || proj) && sc->dev.mb_table) grid = std::min(grid, (int)(sc->dev.mb_threads / kCtaThreads));
    const uint32_t rec4 = 2 + 2 * ((sc->dev.dim + 3) / 4);
    QueueDev q;
    memset(&q, 0, sizeof q);
    q.capacity = sc->queue_capacity; q.rec4 = rec4;
    q.in = nullptr;
    q.out = sc->d_queue[0];
    q.out_count = d_ctl + CTL_COUNT0 + 1;
    q.in_count = q.in_cursor = nullptr;
    if (tgt.out_mode != NTR_OUT_IDS && !rays) {   // the hit-id hook and a batch of rays leave the last frame's refine mask alone
        sc->last = {};
        sc->last.valid = true; sc->last.adaptive = adaptive;
        sc->last.win_w = win_w; sc->last.win_h = win_h; sc->last.out_rows = f.out_rows;
        sc->last.trf = tile_row_first; sc->last.trs = f.tile_row_step; sc->last.compact = compact;
        sc->last.halo = adaptive ? count_halo(f) : 0;
    }
    auto mark = [&]() {
        if (!(sc->pass_timing || passes) || sc->n_pass_ev >= kMaxPasses + 4) return;
        if (!sc->pass_ev[sc->n_pass_ev]) cudaEventCreate(&sc->pass_ev[sc->n_pass_ev]);
        cudaEventRecord(sc->pass_ev[sc->n_pass_ev++], st);
    };
    sc->n_pass_ev = 0;
    mark();
    if (rays) {
        // the ray-fed primary pass: per lane, non-wide, one build per FLAGS & 3; no more CTAs than the exact mailbox has columns
        const int rf = flags & (NTR_F_GENERAL | NTR_F_COUNT);
        if (!sc->rays_grid[rf]) sc->rays_grid[rf] = std::max(1, sc->kset(rf)->rays_blocks_per_sm()) * sc->sm_count;
        int rgrid = sc->rays_grid[rf];
        if (sc->dev.mb_table) rgrid = std::min(rgrid, (int)(sc->dev.mb_threads / kCtaThreads));
        QueueDev qr = q;
        if (!passes) qr.out = nullptr;
        sc->kset(rf)->render_rays(dim3(rgrid), dim3(kCtaThreads), st, sc->dev, f, qr, ctl, tgt.ray_o, tgt.ray_d, (uint32_t)win_w);
    } else {
        ks->render_pass(dim3(grid), dim3(kCtaThreads), st, sc->dev, sc->cam, f, q, ctl);
    }
    ++sc->launches;
    mark();
#if NTR_FETCH_STATS
    dump_stats("primary", 0);
#endif
    if (use_sched) {
        // schedule for the next frame of this view, computed on the device right behind the primary pass
        const int tb = (int)((n_tiles + 127) / 128);
        order_tiles_kernel<<<tb, 128, 0, st>>>(sc->d_tile_cost[slot], sc->d_tile_order[slot], (uint32_t)n_tiles);
        decay_tile_cost_kernel<<<tb, 128, 0, st>>>(sc->d_tile_cost[slot], (uint32_t)n_tiles);
        sc->launches += 2;
        sc->sched_ready[slot] = true;
    }
    // the list-driven primary passes of an adaptive frame: per-lane, non-wide NTR_F_LIST builds; no more CTAs than the
    // exact mailbox has columns
    const int lflags = (flags & (NTR_F_GENERAL | NTR_F_COUNT)) | NTR_F_LIST | (proj ? NTR_F_PROJ : 0);
    auto list_pass = [&](const FrameDev &fl, uint32_t *cursor, QueueDev ql) {
        ControlDev cl = ctl;
        cl.tile_cursor = cursor;
        if (!passes) ql.out = nullptr;
        int lgrid = grid_for(sc, lflags);
        if (sc->dev.mb_table) lgrid = std::min(lgrid, (int)(sc->dev.mb_threads / kCtaThreads));
        sc->kset(lflags)->render_pass(dim3(lgrid), dim3(kCtaThreads), st, sc->dev, sc->cam, fl, ql, cl);
        ++sc->launches;
    };
    if (adaptive && sc->last.halo) {
        // the corner pixels of the mask that this launch does not own, at factor 1; their bounces join the base frame's
        FrameDev fh = f;
        fh.list_n = (uint32_t)nhalo;
        list_pass(fh, d_ctl + CTL_HALO_CURSOR, q);
        mark();
    }
    // one round of bounce passes: queue counters at cnt0 + depth, cursors at cur0 + depth, sort sizes from prev[depth]
    auto bounces = [&](int cnt0, int cur0, const uint32_t *prev) -> int {
        for (int depth = 1; depth <= sc->dev.max_depth; ++depth) {
            q.in = sc->d_queue[(depth - 1) & 1];
            q.out = sc->d_queue[depth & 1];
            q.in_count = d_ctl + cnt0 + depth;
            q.out_count = d_ctl + cnt0 + depth + 1;
            q.in_cursor = d_ctl + cur0 + depth;
            q.in_perm = nullptr;
            q.n_sorted = 0;
            q.ring_start = nullptr;
            // adaptive: the sort (one read-back + key kernel + radix sort per pass) only pays for expensive rays; cheap scenes
            // (config 3: 0.45 ns/ray) lose 20 % to it, star polytopes (6-16 ns/ray unsorted) gain 26-29 %
            if (sc->sort_rays && pass_ns_per_ray > 1.5f && prev[depth] >= (1u << 15)) {
                // Re-bin the bounces for coherence: reflection rays get more divergent with every depth (measured on
                // config 4: 1.5 ns/ray for primaries, 6 -> 16 ns/ray for depths 1 -> 4).  Sorting them by a key made of
                // direction signs + quantised direction + quantised origin hands every warp 32 rays that walk the same
                // part of the tree.  The sort size is the count this pass had in the previous frame plus a margin (no
                // read-back between the passes; see ray_keys_kernel).
                const uint32_t n = (uint32_t)std::min<uint64_t>((uint64_t)prev[depth] + prev[depth] / 8 + 4096, sc->queue_capacity);
                if (sc->sort_cap < n) {
                    for (int k = 0; k < 2; ++k) { cudaFree(sc->d_keys[k]); cudaFree(sc->d_perm[k]); sc->d_keys[k] = sc->d_perm[k] = nullptr; }
                    cudaFree(sc->d_sort_tmp); sc->d_sort_tmp = nullptr; sc->sort_cap = 0;
                    const uint32_t cap = n + n / 4;
                    for (int k = 0; k < 2; ++k) {
                        CUDA_TRY(cudaMalloc(&sc->d_keys[k], (size_t)cap * 4));
                        CUDA_TRY(cudaMalloc(&sc->d_perm[k], (size_t)cap * 4));
                    }
                    size_t bytes = 0;
                    cub::DeviceRadixSort::SortPairs(nullptr, bytes, sc->d_keys[0], sc->d_keys[1], sc->d_perm[0], sc->d_perm[1], (int)cap);
                    CUDA_TRY(cudaMalloc(&sc->d_sort_tmp, bytes));
                    sc->sort_tmp_bytes = bytes;
                    sc->sort_cap = cap;
                }
                ray_keys_kernel<<<(n + 255) / 256, 256, 0, st>>>(q.in, rec4, n, q.in_count, sc->queue_capacity, sc->dev.dim, sc->dev,
                                                                   sc->d_keys[0], sc->d_perm[0], sc->heavy_first ? 1 : 0);
                size_t bytes = sc->sort_tmp_bytes;
                cub::DeviceRadixSort::SortPairs(sc->d_sort_tmp, bytes, sc->d_keys[0], sc->d_keys[1], sc->d_perm[0], sc->d_perm[1], (int)n, 0, 32, st);
                sc->launches += 2;
                q.in_perm = sc->d_perm[1];
                q.n_sorted = n;
                if (sc->heavy_first && sc->adaptive_fetch) {
                    if (!sc->d_ring) CUDA_TRY(cudaMalloc(&sc->d_ring, (kMaxPasses + 2) * 4 * sizeof(uint32_t)));
                    uint32_t *ring = sc->d_ring + (size_t)depth * 4;
                    CUDA_TRY(cudaMemsetAsync(ring, 0xFF, 4 * sizeof(uint32_t), st));
                    ring_bounds_kernel<<<(n + 255) / 256, 256, 0, st>>>(sc->d_keys[1], n, q.in_count, sc->queue_capacity, ring);
                    ++sc->launches;
                    q.ring_start = ring;
                    q.fetch_sizes = sc->fetch_sizes;
                }
            }
            const int bf = bounce_flags | wide_for(depth < 32 ? depth : 31);
            sc->kset(bf)->render_pass(dim3(grid_for(sc, bf)), dim3(kCtaThreads), st, sc->dev, sc->cam, f, q, ctl);
            ++sc->launches;
            mark();
#if NTR_FETCH_STATS
            dump_stats("bounce", depth);
#endif
        }
        return NTR_OK;
    };
    if (passes) {
        const int rc = bounces(CTL_COUNT0, CTL_CURSOR0, rays ? sc->rays_prev_pass_count : n_views ? sc->views_prev_pass_count
                                                        : proj ? sc->proj_prev_pass_count : sc->prev_pass_count);
        if (rc) return rc;
    }
    if (adaptive) {
        // classify the plain frame: mask and row-major list of the pixels to refine; their count stays on the device
        int rc = ensure((void **)&sc->d_mask, &sc->mask_cap, std::max<size_t>(npix, 1));
        if (!rc) rc = ensure((void **)&sc->d_list, &sc->list_cap, std::max<size_t>(npix, 1) * sizeof(uint32_t));
        if (rc) return rc;
        size_t bytes = 0;
        thrust::counting_iterator<uint32_t> slots(0);
        CUDA_TRY(cub::DeviceSelect::Flagged(nullptr, bytes, slots, sc->d_mask, sc->d_list, d_ctl + CTL_REFINED, (int)npix, st));
        if ((rc = ensure(&sc->d_select_tmp, &sc->select_tmp_cap, std::max<size_t>(bytes, 256)))) return rc;
        const int blocks = (int)std::min<long long>(((long long)npix + 255) / 256, (long long)sc->sm_count * 8);
        if (npix) classify_kernel<<<blocks, 256, 0, st>>>(f, sc->ss_threshold, sc->d_mask);
        bytes = sc->select_tmp_cap;
        CUDA_TRY(cub::DeviceSelect::Flagged(sc->d_select_tmp, bytes, slots, sc->d_mask, sc->d_list, d_ctl + CTL_REFINED, (int)npix, st));
        sc->launches += 2;
        // refine: the listed pixels at factor s over their slots, in a second round of passes of their own
        FrameDev fr = f;
        fr.ss = sc->ss;
        fr.width = width * fr.ss; fr.height = height * fr.ss;
        fr.half_w = (float)fr.width / 2.0f;
        fr.half_h = (float)fr.height / 2.0f;
        fr.fovI = tanf(sc->dev.fov / 2) / fr.half_w;
        if (proj) fr.proj_k = projection_k(sc->proj, sc->proj_param, fr.half_w);
        fr.list = sc->d_list;
        fr.list_count = d_ctl + CTL_REFINED;
        QueueDev qr;
        memset(&qr, 0, sizeof qr);
        qr.capacity = sc->queue_capacity; qr.rec4 = rec4;
        qr.out = sc->d_queue[0];
        qr.out_count = d_ctl + CTL_COUNT0B + 1;
        list_pass(fr, d_ctl + CTL_LIST_CURSOR, qr);
        mark();
        if (passes && (rc = bounces(CTL_COUNT0B, CTL_CURSOR0B, proj ? sc->proj_prev_pass_count2 : sc->prev_pass_count2))) return rc;
    }
    if ((passes || adaptive) && tgt.out_mode == NTR_OUT_PACKED) {
        f.out_mode = NTR_OUT_PACKED;
        const long long groups = (long long)((win_w + 3) / 4) * f.out_rows * (long long)nv;
        const int blocks = (int)std::min<long long>((groups + 255) / 256, (long long)sc->sm_count * 8);
        pack_kernel<<<blocks, 256, 0, st>>>(f);
        ++sc->launches;
    }
    CUDA_TRY(cudaGetLastError());
    if (!sc->frame_done[sc->ctl_slot]) CUDA_TRY(cudaEventCreateWithFlags(&sc->frame_done[sc->ctl_slot], cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(sc->frame_done[sc->ctl_slot], st));
    sc->frame_stream[sc->ctl_slot] = st;
    return NTR_OK;
}

// A device->host copy of the finished frame that run_frame_sync may enqueue right behind the kernels, so that frames
// without wavefront passes need a single stream synchronisation.
struct HostCopy {
    void *dst; size_t dpitch; const void *src; size_t spitch, row_bytes; int rows;
    bool done;
};

// One frame in two halves, so that a caller with several devices can have all of them tracing before it waits for any:
// frame_submit enqueues the kernels and the read-back of the control block (into pinned memory: never blocks),
// frame_collect waits, does the bookkeeping and says whether the frame has to be traced again (a wavefront queue
// overflowed and was regrown).
struct FrameJob {
    int width, height, x0, y0, win_w, win_h;
    const ntr_image_format *fmt;
    RenderTarget tgt;
    int trf, trs, compact;
    cudaStream_t st;
    bool passes = false;
    const CameraDev *views = nullptr;   // a batch of views (device array) and its size; 0: one frame through the scene's camera
    uint32_t n_views = 0;
    bool restart_clock = true;          // false: ev0 keeps marking the start of an earlier launch of the same call
    bool proj = false;                  // the last submit ran under a projection other than the perspective one
};

int frame_submit(ntr_scene *sc, FrameJob &j) {
    if (j.restart_clock) CUDA_TRY(cudaEventRecord(sc->ev0, j.st));
    j.proj = j.tgt.out_mode != NTR_OUT_RAYS && sc->proj != NTR_PROJ_PERSPECTIVE;
    int rc = enqueue_frame(sc, j.st, j.width, j.height, j.x0, j.y0, j.win_w, j.win_h, j.fmt, j.tgt, j.trf, j.trs, j.compact, &j.passes,
                           j.views, j.n_views);
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(sc->ev1, j.st));
    sc->timing_valid = true;
    return NTR_OK;
}

int frame_readback(ntr_scene *sc, FrameJob &j) {
    CUDA_TRY(cudaMemcpyAsync(sc->h_ctl, sc->d_ctl, CTL_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, j.st));
    CUDA_TRY(cudaMemcpyAsync(sc->h_cnt, sc->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, j.st));
    return NTR_OK;
}

int frame_collect(ntr_scene *sc, FrameJob &j, bool *again) {
    *again = false;
    CUDA_TRY(cudaStreamSynchronize(j.st));
    const uint32_t *h_ctl = sc->h_ctl;
    const unsigned long long *h_cnt = sc->h_cnt;
    const bool adaptive = frame_adaptive(sc, j.tgt.out_mode);
    if (j.passes && sc->n_pass_ev > 2) {
        // cost of the wavefront passes per ray: feeds the decision to re-bin rays in the next frame
        float ms = 0;
        cudaEventElapsedTime(&ms, sc->pass_ev[1], sc->pass_ev[sc->n_pass_ev - 1]);
        uint64_t rays = 0;
        for (int d = 1; d <= sc->dev.max_depth && d <= kMaxPasses; ++d) rays += std::min(h_ctl[CTL_COUNT0 + d], sc->queue_capacity);
        if (adaptive)
            for (int d = 1; d <= sc->dev.max_depth && d <= kMaxPasses; ++d) rays += std::min(h_ctl[CTL_COUNT0B + d], sc->queue_capacity);
        if (rays > 0)
            (j.tgt.out_mode == NTR_OUT_RAYS ? sc->rays_pass_ns_per_ray : j.n_views ? sc->views_pass_ns_per_ray
             : j.proj ? sc->proj_pass_ns_per_ray : sc->pass_ns_per_ray) = ms * 1e6f / (float)rays;
    }
    uint32_t *const prev = j.tgt.out_mode == NTR_OUT_RAYS ? sc->rays_prev_pass_count
                           : j.n_views ? sc->views_prev_pass_count : j.proj ? sc->proj_prev_pass_count : sc->prev_pass_count;
    uint32_t *const prev2 = j.proj ? sc->proj_prev_pass_count2 : sc->prev_pass_count2;
    if (j.passes) for (int d = 1; d <= kMaxPasses; ++d) prev[d] = std::min(h_ctl[CTL_COUNT0 + d], sc->queue_capacity);
    if (j.passes && adaptive)
        for (int d = 1; d <= kMaxPasses; ++d) prev2[d] = std::min(h_ctl[CTL_COUNT0B + d], sc->queue_capacity);
    if (sc->pass_timing && sc->n_pass_ev > 1) {
        fprintf(stderr, "ntr pass ms:");
        for (int i = 0; i + 1 < sc->n_pass_ev; ++i) {
            float ms = 0;
            cudaEventElapsedTime(&ms, sc->pass_ev[i], sc->pass_ev[i + 1]);
            fprintf(stderr, " %.3f", ms);
        }
        fprintf(stderr, "  rays:");
        for (int d = 1; d <= sc->dev.max_depth + 1 && d <= kMaxPasses; ++d) fprintf(stderr, " %u", h_ctl[CTL_COUNT0 + d]);
        fprintf(stderr, "\n");
    }
    if (sc->h_abort[sc->abort_idx]) return fail(NTR_ERR_ABORTED, "render aborted");
    const uint64_t overflows = sc->counters.queue_overflows;
    // an adaptive frame traces its own pixels and its halo once, and the refined pixels ss*ss times more
    const uint64_t fss = adaptive ? 1 : (uint64_t)frame_ss(sc, j.tgt.out_mode), spp = fss * fss;
    sc->counters.primary_rays = (uint64_t)j.win_w * j.win_h * spp * (j.n_views ? j.n_views : 1);
    if (j.trs > 1) {
        const int tiles_y = (j.win_h + NTR_TILE - 1) / NTR_TILE;
        uint64_t rows = 0;
        for (int ty = j.trf; ty < tiles_y; ty += j.trs) rows += std::min(NTR_TILE, j.win_h - ty * NTR_TILE);
        sc->counters.primary_rays = rows * (uint64_t)j.win_w * spp;
    }
    if (adaptive) {
        sc->last.refined = h_ctl[CTL_REFINED];
        sc->counters.primary_rays += sc->last.halo + sc->last.refined * (uint64_t)sc->ss * sc->ss;
    }
    sc->counters.reflection_rays = h_cnt[1]; sc->counters.shadow_rays = h_cnt[2]; sc->counters.node_steps = h_cnt[3];
    sc->counters.simplex_tests = h_cnt[4]; sc->counters.solid_tests = h_cnt[5]; sc->counters.shaded_hits = h_cnt[6];
    sc->counters.truncated_hit_lists = h_cnt[7];
    sc->counters.queue_overflows = overflows;
    if (!j.passes || !h_ctl[CTL_OVERFLOW]) return NTR_OK;
    // a wavefront queue was too small: the counters say how many records were wanted
    uint32_t need = 0;
    for (int d = 1; d <= kMaxPasses; ++d) need = std::max(need, std::max(h_ctl[CTL_COUNT0 + d], h_ctl[CTL_COUNT0B + d]));
    sc->counters.queue_overflows = overflows + 1;
    int rc = ensure_queues(sc, (uint32_t)std::min<uint64_t>((uint64_t)need * 2 + 1024, 0x7FFFFFFFu));
    if (rc) return rc;
    *again = true;
    return NTR_OK;
}

// Runs a frame on `st`, waits for it, handles queue overflow (regrow + retry) and abort.
int run_frame_sync(ntr_scene *sc, int width, int height, int x0, int y0, int win_w, int win_h,
                   const ntr_image_format *fmt, const RenderTarget &tgt, int trf, int trs, int compact,
                   cudaStream_t st, HostCopy *hc = nullptr) {
    FrameJob j{width, height, x0, y0, win_w, win_h, fmt, tgt, trf, trs, compact, st};
    for (int attempt = 0; attempt < 8; ++attempt) {
        int rc = frame_submit(sc, j);
        if (rc) return rc;
        if (hc && !j.passes) {            // no overflow / retry possible: the frame in d_packed is final
            CUDA_TRY(cudaMemcpy2DAsync(hc->dst, hc->dpitch, hc->src, hc->spitch, hc->row_bytes, hc->rows, cudaMemcpyDeviceToHost, st));
            hc->done = true;
        }
        if ((rc = frame_readback(sc, j))) return rc;
        bool again = false;
        if ((rc = frame_collect(sc, j, &again))) return rc;
        if (!again) return NTR_OK;
    }
    return fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing");
}

int ensure_stage(ntr_scene *sc, size_t bytes) {
    if (sc->h_stage_cap >= bytes && sc->h_stage) return NTR_OK;
    if (sc->h_stage) { cudaFreeHost(sc->h_stage); sc->h_stage = nullptr; sc->h_stage_cap = 0; }
    CUDA_TRY(cudaHostAlloc((void **)&sc->h_stage, bytes + bytes / 8, cudaHostAllocDefault));
    sc->h_stage_cap = bytes + bytes / 8;
    return NTR_OK;
}

// rows [y0, y1) of the staging buffer -> the caller's buffer; only the pixel bytes are written, like process_pixel: the
// pitch padding of `dst` is left alone
void unstage_rows(const ntr_scene *sc, unsigned char *dst, size_t pitch, size_t row_bytes, int y0, int y1) {
    if (row_bytes == pitch) memcpy(dst + (size_t)y0 * pitch, sc->h_stage + (size_t)y0 * pitch, (size_t)(y1 - y0) * pitch);
    else for (int y = y0; y < y1; ++y) memcpy(dst + (size_t)y * pitch, sc->h_stage + (size_t)y * pitch, row_bytes);
}

// A finished device frame into a PAGEABLE destination: row chunks go device -> pinned staging back to back on `st`, the
// host copies chunk k out of the staging buffer as soon as its event fires -- while chunk k+1 crosses PCIe.
int download_staged(ntr_scene *sc, unsigned char *dst, size_t pitch, size_t row_bytes, int rows, const unsigned char *src, cudaStream_t st) {
    int rc = ensure_stage(sc, pitch * (size_t)rows);
    if (rc) return rc;
    const int chunks = (int)std::min<size_t>(8, std::max<size_t>(1, pitch * (size_t)rows / (1u << 20)));
    for (int c = 0; c < chunks; ++c) {
        if (!sc->stage_ev[c]) CUDA_TRY(cudaEventCreateWithFlags(&sc->stage_ev[c], cudaEventDisableTiming));
        const int y0 = (int)((long long)rows * c / chunks), y1 = (int)((long long)rows * (c + 1) / chunks);
        CUDA_TRY(cudaMemcpy2DAsync(sc->h_stage + (size_t)y0 * pitch, pitch, src + (size_t)y0 * pitch, pitch, row_bytes, y1 - y0, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaEventRecord(sc->stage_ev[c], st));
    }
    for (int c = 0; c < chunks; ++c) {
        const int y0 = (int)((long long)rows * c / chunks), y1 = (int)((long long)rows * (c + 1) / chunks);
        CUDA_TRY(cudaEventSynchronize(sc->stage_ev[c]));
        unstage_rows(sc, dst, pitch, row_bytes, y0, y1);
    }
    return NTR_OK;
}

// ntr_render for frames that need a single pass, into a pinned destination: slabs of tile rows, each with its own
// persistent kernel and device->host copy on its own stream.  The kernels queue up behind each other on the device
// (each fills the machine; the next one's CTAs move in as the previous one's retire, so no tail is added) and the copy
// of slab k runs while slab k+1 is traced.  Returns 1 when it does not apply (the caller uses the plain path).
// `staged`: the destination is pageable -- the slabs land in the pinned staging buffer and the host copies slab k out
// while slab k+1 is traced and transferred.
int run_frame_slabs(ntr_scene *sc, const ntr_image_format *fmt, unsigned char *dst, bool staged) {
    const int tiles_y = (fmt->height + NTR_TILE - 1) / NTR_TILE;
    const int S = std::min(kSlabMax, tiles_y / 4);
    // (the slabs' kernels run side by side: they would share the columns of the exact mailbox table)
    if (S < 2 || sc->instrumented || sc->dev.mb_table) return 1;
    for (int i = 0; i < S; ++i) {
        if (i && !sc->slab_stream[i]) CUDA_TRY(cudaStreamCreateWithFlags(&sc->slab_stream[i], cudaStreamNonBlocking));
        if (!sc->slab_done[i]) CUDA_TRY(cudaEventCreateWithFlags(&sc->slab_done[i], cudaEventDisableTiming));
    }
    const size_t pitch = (size_t)fmt->pitch, row_bytes = (size_t)fmt->width * fmt->bytes_per_pixel;
    if (staged) { const int rcs = ensure_stage(sc, pitch * (size_t)fmt->height); if (rcs) return rcs; }
    unsigned char *const host = staged ? sc->h_stage : dst;
    int slab_y0[kSlabMax], slab_y1[kSlabMax];
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_PACKED;
    CUDA_TRY(cudaEventRecord(sc->ev0, sc->stream));
    int rc = NTR_OK;
    for (int i = 0; i < S && rc == NTR_OK; ++i) {
        cudaStream_t st = i ? sc->slab_stream[i] : sc->stream;
        if (i) CUDA_TRY(cudaStreamWaitEvent(st, sc->ev0, 0));
        const int y0 = (int)((long long)tiles_y * i / S) * NTR_TILE;
        const int y1 = std::min(fmt->height, (int)((long long)tiles_y * (i + 1) / S) * NTR_TILE);
        tgt.packed = sc->d_packed + (size_t)y0 * pitch;
        slab_y0[i] = y0; slab_y1[i] = y1;
        bool p = false;
        sc->ctl_slot = i;
        rc = enqueue_frame(sc, st, fmt->width, fmt->height, 0, y0, fmt->width, y1 - y0, fmt, tgt, 0, 1, 0, &p);
        sc->ctl_slot = 0;
        if (rc) break;
        // only the pixel bytes are written, like process_pixel: the pitch padding of `dst` is left alone
        CUDA_TRY(cudaMemcpy2DAsync(host + (size_t)y0 * pitch, pitch, tgt.packed, pitch, row_bytes, y1 - y0, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaEventRecord(sc->slab_done[i], st));
    }
    for (int i = 1; i < S; ++i) cudaStreamWaitEvent(sc->stream, sc->slab_done[i], 0);
    if (rc) { cudaStreamSynchronize(sc->stream); return rc; }
    sc->last.win_h = fmt->height; sc->last.out_rows = fmt->height;      // the refine mask covers the whole (plain) frame
    CUDA_TRY(cudaEventRecord(sc->ev1, sc->stream));
    sc->timing_valid = true;
    if (staged) {
        for (int i = 0; i < S; ++i) {           // slab i leaves the staging buffer while the later ones are traced / in flight
            CUDA_TRY(cudaEventSynchronize(sc->slab_done[i]));
            unstage_rows(sc, dst, pitch, row_bytes, slab_y0[i], slab_y1[i]);
        }
    }
    unsigned long long h_cnt[kSlabMax * 8];
    CUDA_TRY(cudaMemcpyAsync(h_cnt, sc->d_counters, sizeof(unsigned long long) * 8 * S, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    if (sc->h_abort[0]) return fail(NTR_ERR_ABORTED, "render aborted");
    const uint64_t overflows = sc->counters.queue_overflows;
    sc->counters = ntr_counters{};
    sc->counters.queue_overflows = overflows;
    sc->counters.primary_rays = (uint64_t)fmt->width * fmt->height * sc->ss * sc->ss;
    for (int i = 0; i < S; ++i) {
        sc->counters.reflection_rays += h_cnt[i * 8 + 1]; sc->counters.shadow_rays += h_cnt[i * 8 + 2];
        sc->counters.shaded_hits += h_cnt[i * 8 + 6]; sc->counters.truncated_hit_lists += h_cnt[i * 8 + 7];
    }
    return NTR_OK;
}

struct BusyGuard {
    ntr_scene *sc;
    bool ok;
    explicit BusyGuard(ntr_scene *s) : sc(s), ok(!s->busy.exchange(true)) { if (ok) { s->h_abort[0] = 0; s->abort_idx = 0; } }
    ~BusyGuard() { if (ok) sc->busy.store(false); }
};

#define ENTER(sc)                                                                               \
    if (!(sc)) return fail(NTR_ERR_VALUE, "scene is NULL");                                     \
    CUDA_TRY(cudaSetDevice((sc)->device));                                                      \
    BusyGuard guard_(sc);                                                                       \
    if (!guard_.ok) return fail(NTR_ERR_RUNTIME, "the renderer is already running")

// accum (3 floats per window pixel) -> packed image.  One thread packs 4 consecutive pixels of a row so the
// 4*bpp bytes it owns are a whole number of 32-bit words.
// A batch of views packs all its frames: accumulator row v * out_rows + y is row y of frame v (at packed + v * pitch * win_h).
__global__ void pack_kernel(const __grid_constant__ FrameDev f) {
    const int groups_x = (f.win_w + 3) / 4;
    const long long total = (long long)groups_x * f.out_rows * (f.n_views ? f.n_views : 1);
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total; g += (long long)gridDim.x * blockDim.x) {
        const long long ya = g / groups_x;          // accumulator row
        const int x0 = (int)(g % groups_x) * 4;
        const int y = (int)(ya % f.out_rows);
        const long long view = ya / f.out_rows;
        if (!f.compact && f.tile_row_step > 1) {
            // interleaved render at frame positions: the rows of the other ranks' tile rows are not this rank's to write
            const int ty = y / NTR_TILE;
            if (ty < f.tile_row_first || (ty - f.tile_row_first) % f.tile_row_step != 0) continue;
        }
        const int n = min(4, f.win_w - x0);
        const int bpp = f.fmt.bytes_per_pixel;
        __align__(16) unsigned char buf[64];
        for (int k = 0; k < n; ++k) {
            const float *a = f.accum + ((size_t)ya * f.win_w + x0 + k) * 3;
            const float rgb[3] = {a[0], a[1], a[2]};
            uint32_t w[4];
            pack_pixel(f.fmt, rgb, w);
            for (int j = 0; j < bpp; ++j) {
                const int sj = f.fmt.reversed ? bpp - 1 - j : j;
                buf[k * bpp + j] = (unsigned char)(w[sj >> 2] >> (8 * (3 - (sj & 3))));
            }
        }
        unsigned char *dst = f.packed + (size_t)view * f.fmt.pitch * f.win_h + (size_t)y * f.fmt.pitch + (size_t)x0 * bpp;
        const int nb = n * bpp;
        if (((size_t)dst & 3) == 0 && (nb & 3) == 0) {
            for (int j = 0; j < nb; j += 4) *(uint32_t *)(dst + j) = *(const uint32_t *)(buf + j);
        } else {
            for (int j = 0; j < nb; ++j) dst[j] = buf[j];
        }
    }
}

// Refine mask of the pixels an adaptive frame owns (trace_core.cuh: refine_pixel), f: the plain frame in the accumulator
__global__ void classify_kernel(const __grid_constant__ FrameDev f, float threshold, unsigned char *mask) {
    const long long npix = (long long)f.win_w * f.out_rows;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < npix; i += (long long)gridDim.x * blockDim.x) {
        const int wx = (int)(i % f.win_w), wy = window_row(f, (int)(i / f.win_w));
        int r = 0;
        mask[i] = owned_row(f, wy, &r) && refine_pixel(f, f.accum, wx, wy, threshold) ? 1 : 0;
    }
}

// Sort key of a queued bounce: [direction signs, 1 bit x K][direction magnitude, 2 bits x K][origin cell, 3 bits x K]
// over the first K = min(D, 5) axes (30 bits).
// With heavy_first the two top bits (30, 31) hold the ray's closest approach to the centre of the scene box, nearest
// first: on star polytopes the rays through the middle walk the giant leaves and cost 10-40x the mean
// (tools/ray_cost_map.py), and a pass that starts them first ends when its bulk ends instead of one heavy ray later
// (tools/sim_schedule.py).  Any order is a valid order: this only changes when a ray is traced, never what it returns.
// `n` is the host's ESTIMATE of the pass size (the count of the same pass in the previous frame plus a margin), so that
// no read-back sits between the passes of a frame; the real count is *count.  Slots beyond it get the largest key and,
// the sort being stable, end up behind every real record; records beyond the estimate are read unsorted (kernels.cuh).
__global__ void ray_keys_kernel(const float4 *recs, uint32_t rec4, uint32_t n, const uint32_t *count, uint32_t capacity, int D,
                                const __grid_constant__ SceneDev s, uint32_t *keys, uint32_t *idx, int heavy_first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i >= min(*count, capacity)) { keys[i] = 0xFFFFFFFFu; idx[i] = i; return; }
    const int K = D < 5 ? D : 5;
    const int D4 = (int)(rec4 - 2) / 2;
    const float *o = reinterpret_cast<const float *>(recs + (size_t)i * rec4 + 2);
    const float *d = reinterpret_cast<const float *>(recs + (size_t)i * rec4 + 2 + D4);
    float len = 0;
    for (int a = 0; a < D; ++a) len += d[a] * d[a];
    len = rsqrtf(fmaxf(len, 1e-30f));
    uint32_t ks = 0, kd = 0, ko = 0;
    for (int a = 0; a < K; ++a) {
        const float da = d[a] * len;
        ks = (ks << 1) | (da < 0 ? 1u : 0u);
        kd = (kd << 2) | (uint32_t)fminf(fabsf(da) * 4.0f, 3.0f);
        const float ext = s.bmax[a] - s.bmin[a];
        const float u = ext > 0 ? (o[a] - s.bmin[a]) / ext : 0.0f;
        ko = (ko << 3) | (uint32_t)fminf(fmaxf(u * 8.0f, 0.0f), 7.0f);
    }
    uint32_t key = (ks << (5 * K)) | (kd << (3 * K)) | ko;
    if (heavy_first) {
        float oc = 0, od = 0, r2 = 0;
        for (int a = 0; a < D; ++a) {
            const float c = 0.5f * (s.bmin[a] + s.bmax[a]), e = 0.5f * (s.bmax[a] - s.bmin[a]);
            const float v = o[a] - c;
            oc += v * v; od += v * d[a] * len; r2 += e * e;
        }
        const float miss2 = fmaxf(oc - od * od, 0.0f) / fmaxf(r2, 1e-30f);      // (closest approach / box radius)^2
        const uint32_t ring = miss2 < 0.01f ? 0u : miss2 < 0.05f ? 1u : miss2 < 0.2f ? 2u : 3u;
        key = (key & 0x3FFFFFFFu) | (ring << 30);
    }
    keys[i] = key;
    idx[i] = i;
}

// First sorted index of cost rings 1..3 (the two top key bits, heavy-first sort): ring_start[1..3], preset to 0xFFFFFFFF.
__global__ void ring_bounds_kernel(const uint32_t *sorted_keys, uint32_t n, const uint32_t *count, uint32_t capacity, uint32_t *ring_start) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t valid = min(min(*count, capacity), n);
    if (i >= valid) return;
    const uint32_t r = sorted_keys[i] >> 30, rp = i ? sorted_keys[i - 1] >> 30 : 0u;
    for (uint32_t k = rp + 1; k <= r; ++k) atomicMin(ring_start + k, i);
}

__global__ void fma_peak_kernel(float *out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const float b = 1.0000001f, c = 1e-7f;
    for (int i = 0; i < iters; ++i) {
        a0 = fmaf(a0, b, c); a1 = fmaf(a1, b, c); a2 = fmaf(a2, b, c); a3 = fmaf(a3, b, c);
        a4 = fmaf(a4, b, c); a5 = fmaf(a5, b, c); a6 = fmaf(a6, b, c); a7 = fmaf(a7, b, c);
    }
    const float s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678f) out[0] = s;
}

}  // namespace

extern "C" {

NTR_API int ntr_abi_version(void) { return NTR_ABI_VERSION; }
NTR_API const char *ntr_last_error(void) { return g_err.c_str(); }

NTR_API int ntr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
    }
    return ok;
}

NTR_API int ntr_scene_create(const ntr_scene_desc *desc, int device, ntr_scene **out) {
    if (!out) return fail(NTR_ERR_VALUE, "out is NULL");
    *out = nullptr;
    int depth = 0;
    int rc = validate_desc(desc, &depth);
    if (rc) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(NTR_ERR_NO_DEVICE, "no CUDA device available: ntracer_b200 renders on sm_100a only and has no CPU fallback");
    }
    if (device < 0) CUDA_TRY(cudaGetDevice(&device));
    if (device >= ndev) return fail(NTR_ERR_VALUE, "device %d out of range", device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(NTR_ERR_NO_DEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only (no fallback)", device, prop.major, prop.minor);
    CUDA_TRY(cudaSetDevice(device));
    ntr_scene *sc = new (std::nothrow) ntr_scene();
    if (!sc) return fail(NTR_ERR_MEMORY, "out of memory");
    sc->device = device;
    sc->sm_count = prop.multiProcessorCount;
    sc->pass_timing = getenv("NTR_PASS_TIMING") != nullptr;
    sc->sort_rays = getenv("NTR_NO_RAY_SORT") == nullptr;
    if (const char *zc = getenv("NTR_ZEROCOPY")) sc->zero_copy = atoi(zc) != 0;
    sc->slabs = getenv("NTR_NO_SLABS") == nullptr;
    if (const char *wb = getenv("NTR_WIDE")) sc->wide_mode = atoi(wb) != 0;
    if (const char *ts = getenv("NTR_TILE_SCHED")) { sc->force_tile_sched = atoi(ts) != 0; sc->no_tile_sched = atoi(ts) == 0; }
    for (uint32_t i = 0; desc->kind == NTR_SCENE_COMPOSITE && i < desc->n_nodes; ++i)
        if (desc->nodes[i].meta & NTR_LEAF_FLAG) sc->max_leaf = std::max(sc->max_leaf, desc->nodes[i].w2);
    sc->heavy_first = sc->max_leaf >= 256;
    sc->warp_path = sc->max_leaf >= 256 ? 1 : 0;
    sc->adaptive_fetch = false;         // measured (round 2 call 4): fewer rays per warp from the expensive rings loses everywhere
    if (const char *wp = getenv("NTR_WARP")) sc->warp_path = std::max(0, std::min(2, atoi(wp)));
    if (const char *hf = getenv("NTR_HEAVY_FIRST")) sc->heavy_first = atoi(hf) != 0;
    if (const char *af = getenv("NTR_ADAPTIVE_FETCH")) sc->adaptive_fetch = atoi(af) != 0;
    if (const char *fs = getenv("NTR_FETCH_SIZES")) {
        unsigned a = 4, b = 8, c = 16;
        if (sscanf(fs, "%u,%u,%u", &a, &b, &c) >= 1) {
            auto cl = [](unsigned v) { return v < 1 ? 1u : v > 32 ? 32u : v; };
            sc->fetch_sizes = cl(a) | (cl(b) << 8) | (cl(c) << 16);
        }
    }
    if (const char *qi = getenv("NTR_QUEUE_INIT")) sc->queue_init = (uint32_t)strtoul(qi, nullptr, 10);
    if (const char *vl = getenv("NTR_VIEWS_PER_LAUNCH")) sc->views_per_launch = (uint32_t)strtoul(vl, nullptr, 10);
    if (const char *rl = getenv("NTR_RAYS_PER_LAUNCH")) sc->rays_per_launch = (uint32_t)strtoul(rl, nullptr, 10);
    sc->tree_depth = depth;
    sc->dev.dim = desc->dim;
    sc->dev.kind = desc->kind;
    sc->dev.root = NTR_NULL_NODE;
    sc->dev.batch = 1;
    // the fixed-dimension kernels assume 4-lane batches (compile-time block offsets); other batch sizes of the
    // reference's SIMD flavours (8, 16) go through the run-time-dimension kernels
    // NTR_FORCE_GENERIC=1 is NTracer(dimension, force_generic=True) (lib/ntracer/wrapper.py:112-118): the run-time-dimension family
    const bool force_generic = getenv("NTR_FORCE_GENERIC") != nullptr && atoi(getenv("NTR_FORCE_GENERIC")) != 0;
    sc->kset = kernel_family((force_generic || (desc->kind == NTR_SCENE_COMPOSITE && desc->batch_size != 4 && desc->batch_size != 1)) ? 0 : desc->dim);
    for (int i = 0; i < desc->dim; ++i) { sc->cam.right[i] = i == 0; sc->cam.up[i] = i == 1; sc->cam.fwd[i] = i == 2; }
    auto bail = [&](int code) { ntr_scene_destroy(sc); return code; };
    fill_params(sc->dev, desc);
    if (desc->kind == NTR_SCENE_COMPOSITE) {
        if ((rc = build_arena(sc, desc))) return bail(rc);
        if ((rc = upload_lights(sc, desc))) return bail(rc);
    }
    // the exact mailbox of scenes whose leaves overrun the bounded table (trace_core.cuh: MailboxStore): one column per
    // thread of the persistent grid, zero-initialised (generation 0 is never current)
    {
        const uint64_t keys = (uint64_t)desc->n_simplex + desc->n_solids;
        const char *mbx = getenv("NTR_EXACT_MAILBOX");
        const bool want = mbx ? atoi(mbx) != 0 : sc->max_leaf > NTR_MAILBOX_CAP;
        if (desc->kind == NTR_SCENE_COMPOSITE && (sc->base_flags & NTR_F_GENERAL) && want && keys <= NTR_MAILBOX_MAX_KEYS) {
            int blocks = 0;
            for (int f = 0; f < 8; ++f) if ((f & NTR_F_GENERAL) == (sc->base_flags & NTR_F_GENERAL)) blocks = std::max(blocks, grid_for(sc, f));
            sc->dev.mb_threads = (uint32_t)blocks * kCtaThreads;
            sc->dev.mb_shift = mailbox_key_shift(desc);
            const uint64_t nk = ((uint64_t)desc->n_simplex >> sc->dev.mb_shift) + 1 + desc->n_solids;
            sc->dev.mb_words = (uint32_t)((nk + NTR_MAILBOX_BITS_PER_WORD - 1) / NTR_MAILBOX_BITS_PER_WORD);
            const size_t bytes = (size_t)(sc->dev.mb_words + 1) * sc->dev.mb_threads * sizeof(uint32_t);
            if (cudaMalloc(&sc->dev.mb_table, bytes) != cudaSuccess) {
                cudaGetLastError();
                return bail(fail(NTR_ERR_MEMORY, "out of device memory for the mailbox table (%zu bytes)", bytes));
            }
            cudaMemset(sc->dev.mb_table, 0, bytes);
        }
    }
    auto cu = [&](cudaError_t e, const char *what) {
        if (e == cudaSuccess) return 0;
        return fail(e == cudaErrorMemoryAllocation ? NTR_ERR_MEMORY : NTR_ERR_RUNTIME, "%s failed: %s", what, cudaGetErrorString(e));
    };
    if ((rc = cu(cudaStreamCreateWithFlags(&sc->stream, cudaStreamNonBlocking), "cudaStreamCreate"))) return bail(rc);
    if ((rc = cu(cudaEventCreate(&sc->ev0), "cudaEventCreate"))) return bail(rc);
    if ((rc = cu(cudaEventCreate(&sc->ev1), "cudaEventCreate"))) return bail(rc);
    if ((rc = cu(cudaMalloc(&sc->d_ctl, kSlabMax * CTL_WORDS * sizeof(uint32_t)), "cudaMalloc"))) return bail(rc);
    if ((rc = cu(cudaMalloc(&sc->d_counters, kSlabMax * 8 * sizeof(unsigned long long)), "cudaMalloc"))) return bail(rc);
    if ((rc = cu(cudaHostAlloc(&sc->h_abort, sizeof(int) * (1 + NTR_FRAMES_IN_FLIGHT), cudaHostAllocMapped), "cudaHostAlloc"))) return bail(rc);
    for (int i = 0; i <= NTR_FRAMES_IN_FLIGHT; ++i) sc->h_abort[i] = 0;
    if ((rc = cu(cudaHostAlloc(&sc->h_ctl, CTL_WORDS * sizeof(uint32_t), cudaHostAllocDefault), "cudaHostAlloc"))) return bail(rc);
    if ((rc = cu(cudaHostAlloc(&sc->h_cnt, 8 * sizeof(unsigned long long), cudaHostAllocDefault), "cudaHostAlloc"))) return bail(rc);
    if ((rc = cu(cudaHostGetDevicePointer(&sc->d_abort, sc->h_abort, 0), "cudaHostGetDevicePointer"))) return bail(rc);
    *out = sc;
    return NTR_OK;
}

NTR_API void ntr_scene_destroy(ntr_scene *sc) {
    if (!sc) return;
    cudaSetDevice(sc->device);
    if (sc->stream) cudaStreamSynchronize(sc->stream);
    cudaFree(sc->arena); cudaFree(sc->d_lights); cudaFree(sc->d_ctl); cudaFree(sc->d_counters); cudaFree(sc->dev.mb_table);
    cudaFree(sc->d_accum); cudaFree(sc->d_packed); cudaFree(sc->d_ids); cudaFree(sc->d_dists);
    cudaFree(sc->d_queue[0]); cudaFree(sc->d_queue[1]); cudaFree(sc->d_scratch);
    for (int i = 0; i < kSchedSlots; ++i) { cudaFree(sc->d_tile_cost[i]); cudaFree(sc->d_tile_order[i]); }
    cudaFree(sc->d_views);
    cudaFree(sc->d_ring);
    cudaFree(sc->d_keys[0]); cudaFree(sc->d_keys[1]); cudaFree(sc->d_perm[0]); cudaFree(sc->d_perm[1]); cudaFree(sc->d_sort_tmp);
    cudaFree(sc->d_mask); cudaFree(sc->d_list); cudaFree(sc->d_select_tmp);
    if (sc->copy_stream) { cudaStreamSynchronize(sc->copy_stream); cudaStreamDestroy(sc->copy_stream); }
    for (int i = 0; i < kSlabMax; ++i) {
        if (sc->slab_stream[i]) { cudaStreamSynchronize(sc->slab_stream[i]); cudaStreamDestroy(sc->slab_stream[i]); }
        if (sc->slab_done[i]) cudaEventDestroy(sc->slab_done[i]);
        if (sc->frame_done[i]) cudaEventDestroy(sc->frame_done[i]);
    }
    for (FrameSlot &fs : sc->slots) {
        cudaFree(fs.d_buf);
        if (fs.h_stage) cudaFreeHost(fs.h_stage);
        cudaFree(fs.d_aov);
        if (fs.h_aov) cudaFreeHost(fs.h_aov);
        if (fs.rendered) cudaEventDestroy(fs.rendered);
        if (fs.copied) cudaEventDestroy(fs.copied);
    }
    if (sc->h_abort) cudaFreeHost(sc->h_abort);
    if (sc->h_stage) cudaFreeHost(sc->h_stage);
    for (cudaEvent_t e : sc->stage_ev) if (e) cudaEventDestroy(e);
    if (sc->h_ctl) cudaFreeHost(sc->h_ctl);
    if (sc->h_cnt) cudaFreeHost(sc->h_cnt);
    if (sc->ev0) cudaEventDestroy(sc->ev0);
    if (sc->ev1) cudaEventDestroy(sc->ev1);
    if (sc->stream) cudaStreamDestroy(sc->stream);
    cudaGetLastError();
    delete sc;
}

NTR_API int ntr_scene_set_camera(ntr_scene *sc, const float *origin, const float *axes) {
    if (!sc || !origin || !axes) return fail(NTR_ERR_VALUE, "NULL argument");
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the scene is locked while rendering");
    const int D = sc->dev.dim;
    for (int i = 0; i < D; ++i) {
        sc->cam.origin[i] = origin[i];
        sc->cam.right[i] = axes[i]; sc->cam.up[i] = axes[D + i]; sc->cam.fwd[i] = axes[2 * D + i];
    }
    return NTR_OK;
}

NTR_API int ntr_scene_set_supersampling(ntr_scene *sc, int factor) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    if (factor < 1 || factor > NTR_MAX_SUPERSAMPLING) return fail(NTR_ERR_VALUE, "the supersampling factor must be between 1 and %d", NTR_MAX_SUPERSAMPLING);
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the scene is locked while rendering");
    sc->ss = factor;
    return NTR_OK;
}

NTR_API int ntr_scene_set_supersampling_threshold(ntr_scene *sc, float threshold) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    if (isnan(threshold) || threshold == INFINITY) return fail(NTR_ERR_VALUE, "the supersampling threshold must be a finite number (negative: off)");
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the scene is locked while rendering");
    sc->ss_threshold = threshold < 0.0f ? -1.0f : threshold;
    return NTR_OK;
}

static int check_projection(int kind, float param) {
    if (kind == NTR_PROJ_PERSPECTIVE) return NTR_OK;
    if (kind == NTR_PROJ_ORTHOGRAPHIC) {
        if (!(param > 0.0f && param < INFINITY)) return fail(NTR_ERR_VALUE, "the orthographic half width must be finite and positive");
        return NTR_OK;
    }
    if (kind == NTR_PROJ_EQUIRECTANGULAR) {
        if (!(param > 0.0f && param <= 6.283185307179586f))     // 2 pi, rounded to float
            return fail(NTR_ERR_VALUE, "the equirectangular field angle must lie in (0, 2*pi] radians");
        return NTR_OK;
    }
    return fail(NTR_ERR_VALUE, "unknown projection kind %d", kind);
}

NTR_API int ntr_scene_set_projection(ntr_scene *sc, int kind, float param) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    int rc = check_projection(kind, param);
    if (rc) return rc;
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the scene is locked while rendering");
    sc->proj = kind;
    sc->proj_param = kind == NTR_PROJ_PERSPECTIVE ? 0.0f : param;
    return NTR_OK;
}

NTR_API int ntr_last_refine_mask(ntr_scene *sc, uint8_t *mask, size_t len, uint64_t *count) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    if (!sc->last.valid) return fail(NTR_ERR_RUNTIME, "nothing has been rendered yet");
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the renderer is running");
    const auto &L = sc->last;
    if (mask) {
        if (len < (size_t)L.win_w * L.win_h) return fail(NTR_ERR_VALUE, "the mask of the last frame needs %d x %d bytes", L.win_w, L.win_h);
        std::vector<unsigned char> h;
        if (L.adaptive) {
            h.resize((size_t)L.win_w * L.out_rows);
            CUDA_TRY(cudaSetDevice(sc->device));
            CUDA_TRY(cudaMemcpy(h.data(), sc->d_mask, h.size(), cudaMemcpyDeviceToHost));
        }
        FrameDev g;
        memset(&g, 0, sizeof g);
        g.win_w = L.win_w; g.win_h = L.win_h; g.tiles_y = (L.win_h + NTR_TILE - 1) / NTR_TILE;
        g.tile_row_first = L.trf; g.tile_row_step = L.trs; g.compact = L.compact;
        for (int wy = 0, r = 0; wy < L.win_h; ++wy) {
            if (!owned_row(g, wy, &r)) continue;
            unsigned char *row = mask + (size_t)wy * L.win_w;
            if (L.adaptive) memcpy(row, h.data() + (size_t)r * L.win_w, (size_t)L.win_w);
            else memset(row, 0, (size_t)L.win_w);
        }
    }
    if (count) *count = L.adaptive ? L.refined : 0;
    return NTR_OK;
}

NTR_API int ntr_scene_set_params(ntr_scene *sc, const ntr_scene_desc *desc) {
    if (!sc || !desc) return fail(NTR_ERR_VALUE, "NULL argument");
    if (sc->busy) return fail(NTR_ERR_RUNTIME, "the scene is locked while rendering");
    if (desc->dim != sc->dev.dim || desc->kind != sc->dev.kind) return fail(NTR_ERR_VALUE, "dimension / kind mismatch");
    CUDA_TRY(cudaSetDevice(sc->device));
    if (desc->kind == NTR_SCENE_COMPOSITE) {
        if (!desc->boundary) return fail(NTR_ERR_VALUE, "composite scene needs a boundary");
        if (desc->bg_gradient_axis < 0 || desc->bg_gradient_axis >= desc->dim) return fail(NTR_ERR_VALUE, "bg_gradient_axis out of range");
        if (desc->max_reflect_depth < 0 || desc->max_reflect_depth > kMaxPasses - 1)
            return fail(NTR_ERR_VALUE, "max_reflect_depth must be between 0 and %d (one wavefront pass per depth)", kMaxPasses - 1);
    }
    fill_params(sc->dev, desc);
    if (desc->kind == NTR_SCENE_COMPOSITE) return upload_lights(sc, desc);
    return NTR_OK;
}

// ntr_render_device and ntr_render without the entry checks (the scene is locked by the caller)
static int render_device_locked(ntr_scene *sc, const ntr_image_format *fmt, void *dev_dst, size_t dst_len, void *stream,
                                int tile_row_first, int tile_row_step, int compact) {
    int rc = check_format(fmt);
    if (rc) return rc;
    if (!dev_dst) return fail(NTR_ERR_VALUE, "destination is NULL");
    if (tile_row_step < 1 || tile_row_first < 0 || tile_row_first >= tile_row_step) return fail(NTR_ERR_VALUE, "bad tile row interleave");
    const int tiles_y = (fmt->height + NTR_TILE - 1) / NTR_TILE;
    const int my_rows = tile_row_first < tiles_y ? (tiles_y - tile_row_first + tile_row_step - 1) / tile_row_step : 0;
    const size_t need = compact ? (size_t)my_rows * NTR_TILE * fmt->pitch : (size_t)fmt->pitch * fmt->height;
    if (dst_len < need) return fail(NTR_ERR_VALUE, "the buffer is too small for an image with the given dimensions");
    cudaStream_t st = stream ? (cudaStream_t)stream : sc->stream;
    const bool composite = sc->dev.kind == NTR_SCENE_COMPOSITE;
    const bool passes = composite && sc->any_reflective && sc->dev.max_depth > 0;
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_PACKED;
    tgt.packed = static_cast<unsigned char *>(dev_dst);
    if (!passes && !frame_adaptive(sc, NTR_OUT_PACKED)) {
        // single persistent kernel, fully asynchronous on the caller's stream
        bool p = false;
        CUDA_TRY(cudaEventRecord(sc->ev0, st));
        rc = enqueue_frame(sc, st, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, tile_row_first,
                           tile_row_step, compact, &p);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(sc->ev1, st));
        sc->timing_valid = true;
        sc->counters = ntr_counters{};
        sc->counters.primary_rays = (uint64_t)fmt->width * fmt->height * sc->ss * sc->ss;
        return NTR_OK;
    }
    // wavefront passes: synchronous on `st` (the queue-overflow check needs the counters back)
    return run_frame_sync(sc, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, tile_row_first,
                          tile_row_step, compact, st);
}

NTR_API int ntr_render_device(ntr_scene *sc, const ntr_image_format *fmt, void *dev_dst, size_t dst_len, void *stream,
                              int tile_row_first, int tile_row_step, int compact) {
    ENTER(sc);
    return render_device_locked(sc, fmt, dev_dst, dst_len, stream, tile_row_first, tile_row_step, compact);
}

static int render_locked(ntr_scene *sc, const ntr_image_format *fmt, void *dst, size_t dst_len) {
    int rc = check_format(fmt);
    if (rc) return rc;
    if (!dst) return fail(NTR_ERR_VALUE, "destination is NULL");
    const size_t bytes = (size_t)fmt->pitch * fmt->height;
    if (dst_len < bytes) return fail(NTR_ERR_VALUE, "the buffer is too small for an image with the given dimensions");
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_PACKED;
    const bool adaptive = frame_adaptive(sc, NTR_OUT_PACKED);
    if (sc->zero_copy && !adaptive && !(sc->dev.kind == NTR_SCENE_COMPOSITE && sc->any_reflective && sc->dev.max_depth > 0)) {
        // Single-pass frame into a pinned (mapped) destination: the packing epilogue of the kernel stores the pixels
        // straight into host memory, so the PCIe transfer runs underneath the tracing instead of after it.
        // MEASURED (B200, PCIe Gen5): byte-identical frames, but SLOWER end to end -- config 1 0.114 -> 0.186 ms,
        // config 2 0.900 -> 0.983 ms, config 3 unchanged: the 24-byte row segments of the 8x4 pixel blocks make poor PCIe
        // writes.  Off unless NTR_ZEROCOPY=1.
        cudaPointerAttributes attr;
        void *mapped = nullptr;
        if (cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost &&
            cudaHostGetDevicePointer(&mapped, dst, 0) == cudaSuccess && mapped) {
            tgt.packed = static_cast<unsigned char *>(mapped);
            return run_frame_sync(sc, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, 0, 1, 0, sc->stream);
        }
        cudaGetLastError();
    }
    if ((rc = ensure((void **)&sc->d_packed, &sc->packed_cap, bytes))) return rc;
    tgt.packed = sc->d_packed;
    // a pinned (or registered) destination is written by the copy engine directly; a pageable one -- what
    // BlockingRenderer.render is normally handed -- goes through the scene's pinned staging buffer in chunks (a plain
    // cudaMemcpy into pageable memory would stage through the driver's bounce buffers, serially)
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const bool staged = !pinned && getenv("NTR_NO_STAGING") == nullptr;
    if (sc->slabs && (pinned || staged) && !adaptive && !(sc->dev.kind == NTR_SCENE_COMPOSITE && sc->any_reflective && sc->dev.max_depth > 0)) {
        rc = run_frame_slabs(sc, fmt, static_cast<unsigned char *>(dst), staged);
        if (rc <= 0) return rc;
    }
    // only the pixel bytes are written, like process_pixel: the pitch padding of `dst` is left alone
    HostCopy hc{dst, (size_t)fmt->pitch, sc->d_packed, (size_t)fmt->pitch, (size_t)fmt->width * fmt->bytes_per_pixel, fmt->height, false};
    if ((rc = run_frame_sync(sc, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, 0, 1, 0, sc->stream, staged ? nullptr : &hc))) return rc;
    if (staged) return download_staged(sc, static_cast<unsigned char *>(dst), hc.dpitch, hc.row_bytes, hc.rows, sc->d_packed, sc->stream);
    if (!hc.done) {
        CUDA_TRY(cudaMemcpy2DAsync(hc.dst, hc.dpitch, hc.src, hc.spitch, hc.row_bytes, hc.rows, cudaMemcpyDeviceToHost, sc->stream));
        CUDA_TRY(cudaStreamSynchronize(sc->stream));
    }
    return NTR_OK;
}

NTR_API int ntr_render(ntr_scene *sc, const ntr_image_format *fmt, void *dst, size_t dst_len) {
    ENTER(sc);
    return render_locked(sc, fmt, dst, dst_len);
}

NTR_API int ntr_render_begin(ntr_scene *sc, const ntr_image_format *fmt, void *dst, size_t dst_len, uint64_t *ticket_out) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    CUDA_TRY(cudaSetDevice(sc->device));
    int rc = check_format(fmt);
    if (rc) return rc;
    if (!dst || !ticket_out) return fail(NTR_ERR_VALUE, "NULL argument");
    const size_t bytes = (size_t)fmt->pitch * fmt->height;
    if (dst_len < bytes) return fail(NTR_ERR_VALUE, "the buffer is too small for an image with the given dimensions");
    const int slot = (int)(sc->next_ticket % NTR_FRAMES_IN_FLIGHT);
    FrameSlot &fs = sc->slots[slot];
    if (fs.open) return fail(NTR_ERR_RUNTIME, "the renderer is already running: %d frames are in flight, end one first", NTR_FRAMES_IN_FLIGHT);
    if (sc->busy.exchange(true)) return fail(NTR_ERR_RUNTIME, "the renderer is already running");
    struct Unbusy { ntr_scene *s; ~Unbusy() { s->busy.store(false); } } unbusy{sc};
    sc->h_abort[1 + slot] = 0;                  // this frame's own word: an earlier abort belongs to the frames it hit
    sc->abort_idx = 1 + slot;
    if (!sc->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&sc->copy_stream, cudaStreamNonBlocking));
    if (!fs.rendered) CUDA_TRY(cudaEventCreateWithFlags(&fs.rendered, cudaEventDisableTiming));
    if (!fs.copied) CUDA_TRY(cudaEventCreateWithFlags(&fs.copied, cudaEventDisableTiming));
    if ((rc = ensure((void **)&fs.d_buf, &fs.d_cap, bytes))) return rc;
    // a pinned (or registered) destination is written by the copy engine directly; anything else goes through staging
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    fs.staged = !pinned;
    if (fs.staged && fs.h_cap < bytes) {
        if (fs.h_stage) { cudaFreeHost(fs.h_stage); fs.h_stage = nullptr; fs.h_cap = 0; }
        CUDA_TRY(cudaHostAlloc((void **)&fs.h_stage, bytes + bytes / 8, cudaHostAllocDefault));
        fs.h_cap = bytes + bytes / 8;
    }
    fs.dst = static_cast<unsigned char *>(dst);
    fs.pitch = (size_t)fmt->pitch;
    fs.row_bytes = (size_t)fmt->width * fmt->bytes_per_pixel;
    fs.height = fmt->height;
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_PACKED;
    tgt.packed = fs.d_buf;
    const bool composite = sc->dev.kind == NTR_SCENE_COMPOSITE;
    const bool passes = composite && sc->any_reflective && sc->dev.max_depth > 0;
    if (!passes && !frame_adaptive(sc, NTR_OUT_PACKED)) {
        // one persistent kernel: fully asynchronous
        bool p = false;
        cudaEventRecord(sc->ev0, sc->stream);
        rc = enqueue_frame(sc, sc->stream, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, 0, 1, 0, &p);
        cudaEventRecord(sc->ev1, sc->stream);
        sc->timing_valid = rc == NTR_OK;
        sc->counters = ntr_counters{};
        sc->counters.primary_rays = (uint64_t)fmt->width * fmt->height * sc->ss * sc->ss;
    } else {
        // wavefront passes need their counters back between passes, an adaptive frame its refined count: traced
        // synchronously, only the copy overlaps
        rc = run_frame_sync(sc, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, 0, 1, 0, sc->stream);
        if (rc == NTR_ERR_ABORTED) rc = NTR_OK;     // reported by ntr_render_end
    }
    if (rc) return rc;
    CUDA_TRY(cudaEventRecord(fs.rendered, sc->stream));
    CUDA_TRY(cudaStreamWaitEvent(sc->copy_stream, fs.rendered, 0));
    unsigned char *host = fs.staged ? fs.h_stage : fs.dst;
    CUDA_TRY(cudaMemcpy2DAsync(host, fs.pitch, fs.d_buf, fs.pitch, fs.row_bytes, fs.height, cudaMemcpyDeviceToHost, sc->copy_stream));
    CUDA_TRY(cudaEventRecord(fs.copied, sc->copy_stream));
    fs.open = true;
    fs.ticket = ++sc->next_ticket;
    *ticket_out = fs.ticket;
    return NTR_OK;
}

NTR_API int ntr_render_end(ntr_scene *sc, uint64_t ticket) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    FrameSlot *fs = nullptr;
    for (FrameSlot &o : sc->slots) {
        if (o.open && o.ticket == ticket) fs = &o;
        else if (o.open && o.ticket < ticket) return fail(NTR_ERR_VALUE, "frames must be ended in the order they were begun");
    }
    if (!fs) return fail(NTR_ERR_VALUE, "no open frame with this ticket");
    CUDA_TRY(cudaSetDevice(sc->device));
    const cudaError_t e = cudaEventSynchronize(fs->copied);
    fs->open = false;
    if (e != cudaSuccess) return fail(NTR_ERR_RUNTIME, "cudaEventSynchronize failed: %s", cudaGetErrorString(e));
    if (sc->h_abort[1 + (int)(fs - sc->slots)]) return fail(NTR_ERR_ABORTED, "render aborted");
    if (fs->staged) {
        // only the pixel bytes are written, like process_pixel: the pitch padding of `dst` is left alone
        if (fs->row_bytes == fs->pitch) memcpy(fs->dst, fs->h_stage, fs->pitch * (size_t)fs->height);
        else for (int y = 0; y < fs->height; ++y) memcpy(fs->dst + (size_t)y * fs->pitch, fs->h_stage + (size_t)y * fs->pitch, fs->row_bytes);
    }
    return NTR_OK;
}

// ---- batches of views (ntr_render_views) ------------------------------------------------------------------------------
// A views call traces its views in launches of at most V views, each one pass per bounce depth over all its views.  V keeps
// the samples of a launch, V * W * H * s^2, at or below kViewsSampleCap = 2^25: the wavefront queues want 2 records per
// traced sample, 2^26 records at the cap, which is the size the queues of a single frame are capped at already
// (enqueue_frame; 4 GB per queue in 4 dimensions); the accumulator then holds at most 2^25 pixels (384 MB) and the device
// frames of a launch V * pitch * H bytes, twice over (one launch is traced while the previous one is copied).
// At 1920x1080 that is 16 views per launch, at 640x480 109.  With AOVs, V also keeps a launch's AOVs, V * W * H * (bytes per
// pixel: 8 + 4 * dim for all three), at or below kViewsAovCap = 1 GB (they are held twice, as the frames are).
// NTR_VIEWS_PER_LAUNCH=n overrides V (tests).
static const uint64_t kViewsSampleCap = 1ull << 25;
static const uint64_t kViewsAovCap = 1ull << 30;

static int views_per_launch(const ntr_scene *sc, const ntr_image_format *fmt, int n, size_t aov_px) {
    const uint64_t npix = (uint64_t)fmt->width * fmt->height, ss = (uint64_t)sc->ss;
    uint64_t v = sc->views_per_launch ? sc->views_per_launch : kViewsSampleCap / (npix * ss * ss);
    if (aov_px && !sc->views_per_launch) v = std::min<uint64_t>(v, kViewsAovCap / (npix * aov_px));
    v = std::min<uint64_t>(v, 0x7FFFFFFFull / npix);        // pixel indices v * npix + pix stay below 2^31
    return (int)std::max<uint64_t>(1, std::min<uint64_t>(v, (uint64_t)n));
}

// camera k of a views call, in the layout of ntr_scene_set_camera
static void view_camera(CameraDev &c, const float *origins, const float *axes, int D, int k) {
    memset(&c, 0, sizeof c);
    const float *o = origins + (size_t)k * D, *a = axes + (size_t)k * D * D;
    for (int i = 0; i < D; ++i) {
        c.origin[i] = o[i];
        c.right[i] = a[i]; c.up[i] = a[D + i]; c.fwd[i] = a[2 * D + i];
    }
}

// the per-frame counters of c added to sum (queue_overflows, a running total of the scene, is the caller's business)
static void add_counters(ntr_counters &sum, const ntr_counters &c) {
    sum.primary_rays += c.primary_rays; sum.reflection_rays += c.reflection_rays; sum.shadow_rays += c.shadow_rays;
    sum.node_steps += c.node_steps; sum.simplex_tests += c.simplex_tests; sum.solid_tests += c.solid_tests;
    sum.shaded_hits += c.shaded_hits; sum.truncated_hit_lists += c.truncated_hit_lists;
}

static int check_views(const ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                       const void *dst, size_t dst_len) {
    int rc = check_format(fmt);
    if (rc) return rc;
    if (n < 1) return fail(NTR_ERR_VALUE, "the number of views must be at least 1");
    if (!origins || !axes || !dst) return fail(NTR_ERR_VALUE, "NULL argument");
    if (dst_len / (size_t)n < (size_t)fmt->pitch * fmt->height)
        return fail(NTR_ERR_VALUE, "the buffer is too small for %d images with the given dimensions", n);
    for (const FrameSlot &fs : sc->slots)
        if (fs.open) return fail(NTR_ERR_RUNTIME, "the renderer is already running: a frame of ntr_render_begin is open");
    return NTR_OK;
}

// the AOV buffers of a views call -> *out (all nullptr for a NULL `aovs`); NTR_ERR_VALUE for a short one
static int check_aovs(int n, const ntr_image_format *fmt, int dim, const ntr_aov_buffers *aovs, AovTarget *out) {
    *out = AovTarget{};
    if (!aovs) return NTR_OK;
    const size_t npix = (size_t)n * fmt->width * fmt->height;
    const void *p[3] = {aovs->ids, aovs->depth, aovs->normals};
    const size_t len[3] = {aovs->ids_len, aovs->depth_len, aovs->normals_len}, per[3] = {1, 1, (size_t)dim};
    static const char *const name[3] = {"ids", "depth", "normals"};
    for (int k = 0; k < 3; ++k) {
        if (!p[k]) continue;
        if (len[k] / per[k] < npix) return fail(NTR_ERR_VALUE, "the %s buffer is too small for %d views", name[k], n);
        out->p[k] = const_cast<void *>(p[k]);
    }
    return NTR_OK;
}

// true when every AOV destination wanted is pinned (or registered) host memory
static bool aovs_pinned(const AovTarget &a) {
    for (int k = 0; k < 3; ++k) {
        if (!a.p[k]) continue;
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, a.p[k]) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (!pinned) return false;
    }
    return true;
}

// One scene's share of a views call: its cameras on the device and its launches.  Frames into host memory (`host`) are traced
// into the device buffer of frame slot k % 2 and cross PCIe on the copy stream while launch k + 1 is traced; a pageable
// destination gets them through the slot's pinned staging buffer, which the host empties while the next launch runs.
// Frames into device memory are stored in place.  The AOVs take the same way as the frames: into the slot's device buffer, then
// across PCIe behind the frames (through the slot's pinned staging buffer when a destination is pageable), or in place.
struct ViewsRun {
    ntr_scene *sc = nullptr;
    const ntr_image_format *fmt = nullptr;
    int n = 0, per = 1;                 // views of the run, views per launch
    unsigned char *dst = nullptr;       // frame 0 of the run
    AovTarget aov;                      // the AOVs of view 0 of the run (none wanted: all nullptr)
    cudaStream_t st = nullptr;
    bool host = false, staged = false, aov_staged = false;
    int done = 0, k = 0;                // views and launches finished
    FrameJob j{};                       // the launch in flight
    int unstage_slot = -1, unstage_first = 0, unstage_n = 0;     // a staged launch whose frames are still to reach dst
    ntr_counters sum{};
    size_t frame_bytes() const { return (size_t)fmt->pitch * fmt->height; }
    size_t frame_pixels() const { return (size_t)fmt->width * fmt->height; }
};

static int views_begin(ViewsRun &r, const float *origins, const float *axes) {
    ntr_scene *sc = r.sc;
    if (r.n < 1) return NTR_OK;
    const size_t aov_px = aov_pixel_bytes(r.aov, sc->dev.dim);
    r.per = views_per_launch(sc, r.fmt, r.n, aov_px);
    std::vector<CameraDev> cams(r.n);
    for (int k = 0; k < r.n; ++k) view_camera(cams[k], origins, axes, sc->dev.dim, k);
    // an asynchronous views call on another stream may still be reading the previous cameras
    if (sc->frame_done[0] && sc->frame_stream[0] != r.st) CUDA_TRY(cudaStreamWaitEvent(r.st, sc->frame_done[0], 0));
    int rc = ensure((void **)&sc->d_views, &sc->views_cap, cams.size() * sizeof(CameraDev));
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(sc->d_views, cams.data(), cams.size() * sizeof(CameraDev), cudaMemcpyHostToDevice, r.st));
    if (!r.host) return NTR_OK;
    if (!sc->copy_stream) CUDA_TRY(cudaStreamCreateWithFlags(&sc->copy_stream, cudaStreamNonBlocking));
    const size_t bytes = (size_t)r.per * r.frame_bytes();
    for (FrameSlot &fs : sc->slots) {
        if (!fs.rendered) CUDA_TRY(cudaEventCreateWithFlags(&fs.rendered, cudaEventDisableTiming));
        if (!fs.copied) CUDA_TRY(cudaEventCreateWithFlags(&fs.copied, cudaEventDisableTiming));
        if ((rc = ensure((void **)&fs.d_buf, &fs.d_cap, bytes))) return rc;
        if (r.staged && fs.h_cap < bytes) {
            if (fs.h_stage) { cudaFreeHost(fs.h_stage); fs.h_stage = nullptr; fs.h_cap = 0; }
            CUDA_TRY(cudaHostAlloc((void **)&fs.h_stage, bytes + bytes / 8, cudaHostAllocDefault));
            fs.h_cap = bytes + bytes / 8;
        }
        const size_t abytes = (size_t)r.per * r.frame_pixels() * aov_px;
        if (abytes && (rc = ensure((void **)&fs.d_aov, &fs.d_aov_cap, abytes))) return rc;
        if (abytes && r.aov_staged && fs.h_aov_cap < abytes) {
            if (fs.h_aov) { cudaFreeHost(fs.h_aov); fs.h_aov = nullptr; fs.h_aov_cap = 0; }
            CUDA_TRY(cudaHostAlloc((void **)&fs.h_aov, abytes, cudaHostAllocDefault));
            fs.h_aov_cap = abytes;
        }
    }
    return NTR_OK;
}

// the frames of the staged launch that was copied last: staging buffer -> dst, pixel bytes only
static int views_unstage(ViewsRun &r) {
    if (r.unstage_slot < 0) return NTR_OK;
    const FrameSlot &fs = r.sc->slots[r.unstage_slot];
    r.unstage_slot = -1;
    CUDA_TRY(cudaEventSynchronize(fs.copied));
    const size_t pitch = (size_t)r.fmt->pitch, row_bytes = (size_t)r.fmt->width * r.fmt->bytes_per_pixel;
    unsigned char *to = r.dst + (size_t)r.unstage_first * r.frame_bytes();
    const size_t rows = (size_t)r.unstage_n * r.fmt->height;
    if (r.staged) {
        if (row_bytes == pitch) memcpy(to, fs.h_stage, rows * pitch);
        else for (size_t y = 0; y < rows; ++y) memcpy(to + y * pitch, fs.h_stage + y * pitch, row_bytes);
    }
    if (r.aov_staged) {
        const int D = r.sc->dev.dim;
        const size_t npix = (size_t)r.unstage_n * r.frame_pixels();
        const AovTarget from = aov_packed(fs.h_aov, r.aov, npix, D), into = aov_offset(r.aov, (size_t)r.unstage_first * r.frame_pixels(), D);
        for (int k = 0; k < 3; ++k) if (into.p[k]) memcpy(into.p[k], from.p[k], npix * aov_bytes(k, D));
    }
    return NTR_OK;
}

// enqueues the next launch (again after an overflow); the host empties the staging buffer of the previous one meanwhile
static int views_submit(ViewsRun &r) {
    ntr_scene *sc = r.sc;
    const int cnt = std::min(r.per, r.n - r.done);
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_PACKED;
    if (r.host) {
        FrameSlot &fs = sc->slots[r.k & 1];
        CUDA_TRY(cudaStreamWaitEvent(r.st, fs.copied, 0));         // the launch before the last one has left the buffer
        tgt.packed = fs.d_buf;
        tgt.aov = aov_packed(fs.d_aov, r.aov, (size_t)cnt * r.frame_pixels(), sc->dev.dim);
    } else {
        tgt.packed = r.dst + (size_t)r.done * r.frame_bytes();
        tgt.aov = aov_offset(r.aov, (size_t)r.done * r.frame_pixels(), sc->dev.dim);
    }
    r.j = FrameJob{r.fmt->width, r.fmt->height, 0, 0, r.fmt->width, r.fmt->height, r.fmt, tgt, 0, 1, 0, r.st};
    r.j.views = sc->d_views + r.done;
    r.j.n_views = (uint32_t)cnt;
    r.j.restart_clock = r.done == 0;
    int rc = frame_submit(sc, r.j);
    if (!rc) rc = frame_readback(sc, r.j);
    if (!rc) rc = views_unstage(r);
    return rc;
}

// waits for the launch in flight; once it needs no retry, sums its counters and sends its frames on their way
static int views_collect(ViewsRun &r, bool *again) {
    ntr_scene *sc = r.sc;
    int rc = frame_collect(sc, r.j, again);
    if (rc || *again) return rc;
    add_counters(r.sum, sc->counters);
    r.sum.queue_overflows = sc->counters.queue_overflows;
    const int cnt = (int)r.j.n_views;
    if (r.host) {
        const int slot = r.k & 1;
        FrameSlot &fs = sc->slots[slot];
        const size_t pitch = (size_t)r.fmt->pitch, row_bytes = (size_t)r.fmt->width * r.fmt->bytes_per_pixel;
        CUDA_TRY(cudaEventRecord(fs.rendered, r.st));
        CUDA_TRY(cudaStreamWaitEvent(sc->copy_stream, fs.rendered, 0));
        unsigned char *to = r.staged ? fs.h_stage : r.dst + (size_t)r.done * r.frame_bytes();
        // only the pixel bytes are written, like process_pixel: the pitch padding of `dst` is left alone
        CUDA_TRY(cudaMemcpy2DAsync(to, pitch, fs.d_buf, pitch, row_bytes, (size_t)cnt * r.fmt->height, cudaMemcpyDeviceToHost, sc->copy_stream));
        const int D = sc->dev.dim;
        const size_t npix = (size_t)cnt * r.frame_pixels();
        const AovTarget from = aov_packed(fs.d_aov, r.aov, npix, D);
        const AovTarget into = r.aov_staged ? aov_packed(fs.h_aov, r.aov, npix, D) : aov_offset(r.aov, (size_t)r.done * r.frame_pixels(), D);
        for (int k = 0; k < 3; ++k)
            if (into.p[k]) CUDA_TRY(cudaMemcpyAsync(into.p[k], from.p[k], npix * aov_bytes(k, D), cudaMemcpyDeviceToHost, sc->copy_stream));
        CUDA_TRY(cudaEventRecord(fs.copied, sc->copy_stream));
        if (r.staged || r.aov_staged) { r.unstage_slot = slot; r.unstage_first = r.done; r.unstage_n = cnt; }
    }
    r.done += cnt;
    ++r.k;
    return NTR_OK;
}

// waits for the last copies (whatever `rc` says, so that nothing lands in dst after the call) and publishes the counters
static int views_finish(ViewsRun &r, int rc) {
    ntr_scene *sc = r.sc;
    if (r.host && sc->copy_stream) {
        const cudaError_t e = cudaStreamSynchronize(sc->copy_stream);
        if (e != cudaSuccess && !rc) rc = fail(NTR_ERR_RUNTIME, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
    }
    if (!rc) rc = views_unstage(r);
    r.unstage_slot = -1;
    if (!rc && r.n > 0) sc->counters = r.sum;
    return rc;
}

// the views of a call on one scene, launch after launch (a queue overflow regrows the queues and traces the launch again)
static int views_run(ViewsRun &r, const float *origins, const float *axes) {
    int rc = views_begin(r, origins, axes);
    for (int attempt = 0; !rc && r.done < r.n;) {
        if (++attempt > 8) { rc = fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing"); break; }
        bool again = false;
        if (!(rc = views_submit(r))) rc = views_collect(r, &again);
        if (!again) attempt = 0;
    }
    return views_finish(r, rc);
}

// The AOVs of view k of an adaptively supersampled views call into `into` (device memory of the scene's device): a one-view
// NTR_F_AOV launch at factor 1 whose frame is thrown away.  The scene's factor, threshold, counters and refine-mask record are
// put back afterwards, so the call's frames, masks and counters are those of the call without AOVs.
static int views_aov_pass(ntr_scene *sc, const float *origins, const float *axes, int k, const ntr_image_format *fmt,
                          const AovTarget &into, cudaStream_t st) {
    const int D = sc->dev.dim;
    int rc = ensure((void **)&sc->d_packed, &sc->packed_cap, (size_t)fmt->pitch * fmt->height);
    if (rc) return rc;
    const int ss = sc->ss;
    const float threshold = sc->ss_threshold;
    const ntr_counters counters = sc->counters;
    const auto last = sc->last;
    sc->ss = 1; sc->ss_threshold = -1.0f;
    ViewsRun r;
    r.sc = sc; r.fmt = fmt; r.n = 1; r.dst = sc->d_packed; r.aov = into; r.st = st;
    rc = views_run(r, origins + (size_t)k * D, axes + (size_t)k * D * D);
    sc->ss = ss; sc->ss_threshold = threshold; sc->counters = counters; sc->last = last;
    return rc;
}

// views_aov_pass for view k into host or device destinations (view 0 of them at `dst`); host ones go through the AOV buffer of
// frame slot 0
static int views_aovs_of(ntr_scene *sc, const float *origins, const float *axes, int k, const ntr_image_format *fmt,
                         const AovTarget &dst, bool device, cudaStream_t st) {
    const int D = sc->dev.dim;
    const size_t npix = (size_t)fmt->width * fmt->height;
    const AovTarget into = aov_offset(dst, (size_t)k * npix, D);
    if (device) return views_aov_pass(sc, origins, axes, k, fmt, into, st);
    FrameSlot &fs = sc->slots[0];
    int rc = ensure((void **)&fs.d_aov, &fs.d_aov_cap, npix * aov_pixel_bytes(dst, D));
    if (rc) return rc;
    const AovTarget scratch = aov_packed(fs.d_aov, dst, npix, D);
    if ((rc = views_aov_pass(sc, origins, axes, k, fmt, scratch, st))) return rc;
    for (int c = 0; c < 3; ++c)
        if (into.p[c]) CUDA_TRY(cudaMemcpyAsync(into.p[c], scratch.p[c], npix * aov_bytes(c, D), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return NTR_OK;
}

// Adaptively supersampled views: one after the other through the single-view route (ntr_render / ntr_render_device), each
// with its camera; the scene's own camera is put back afterwards and the counters are the sums over the views.  AOVs come from
// views_aov_pass, view by view.
static int views_one_by_one(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                            unsigned char *dst, bool device, cudaStream_t st, const AovTarget &aov) {
    const CameraDev saved = sc->cam;
    const size_t fb = (size_t)fmt->pitch * fmt->height;
    ntr_counters sum{};
    int rc = NTR_OK;
    for (int k = 0; k < n && !rc; ++k) {
        view_camera(sc->cam, origins, axes, sc->dev.dim, k);
        rc = device ? render_device_locked(sc, fmt, dst + k * fb, fb, st, 0, 1, 0) : render_locked(sc, fmt, dst + k * fb, fb);
        add_counters(sum, sc->counters);
        sum.queue_overflows = sc->counters.queue_overflows;
        if (!rc && aov.any()) rc = views_aovs_of(sc, origins, axes, k, fmt, aov, device, st);
    }
    sc->cam = saved;
    if (!rc) sc->counters = sum;
    return rc;
}

static int render_views_host(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                             void *dst, size_t dst_len, const ntr_aov_buffers *aovs) {
    int rc = check_views(sc, n, origins, axes, fmt, dst, dst_len);
    AovTarget aov;
    if (!rc) rc = check_aovs(n, fmt, sc->dev.dim, aovs, &aov);
    if (rc) return rc;
    if (frame_adaptive(sc, NTR_OUT_PACKED))
        return views_one_by_one(sc, n, origins, axes, fmt, static_cast<unsigned char *>(dst), false, sc->stream, aov);
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    ViewsRun r;
    r.sc = sc; r.fmt = fmt; r.n = n; r.dst = static_cast<unsigned char *>(dst); r.st = sc->stream;
    r.host = true; r.staged = !pinned;
    r.aov = aov; r.aov_staged = aov.any() && !aovs_pinned(aov);
    return views_run(r, origins, axes);
}

NTR_API int ntr_render_views(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                             void *dst, size_t dst_len) {
    ENTER(sc);
    return render_views_host(sc, n, origins, axes, fmt, dst, dst_len, nullptr);
}

NTR_API int ntr_render_views_aovs(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                                  void *dst, size_t dst_len, const ntr_aov_buffers *aovs) {
    ENTER(sc);
    return render_views_host(sc, n, origins, axes, fmt, dst, dst_len, aovs);
}

static int render_views_device(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                               void *dev_dst, size_t dst_len, const ntr_aov_buffers *aovs, void *stream) {
    int rc = check_views(sc, n, origins, axes, fmt, dev_dst, dst_len);
    AovTarget aov;
    if (!rc) rc = check_aovs(n, fmt, sc->dev.dim, aovs, &aov);
    if (rc) return rc;
    cudaStream_t st = stream ? (cudaStream_t)stream : sc->stream;
    if (frame_adaptive(sc, NTR_OUT_PACKED))
        return views_one_by_one(sc, n, origins, axes, fmt, static_cast<unsigned char *>(dev_dst), true, st, aov);
    ViewsRun r;
    r.sc = sc; r.fmt = fmt; r.n = n; r.dst = static_cast<unsigned char *>(dev_dst); r.st = st; r.aov = aov;
    const bool passes = sc->dev.kind == NTR_SCENE_COMPOSITE && sc->any_reflective && sc->dev.max_depth > 0;
    if (passes) return views_run(r, origins, axes);         // synchronous on `st`, as ntr_render_device with passes
    // single-pass views: every launch fully asynchronous on the caller's stream
    if ((rc = views_begin(r, origins, axes))) return rc;
    CUDA_TRY(cudaEventRecord(sc->ev0, st));
    for (int first = 0; first < n; first += r.per) {
        const int cnt = std::min(r.per, n - first);
        RenderTarget tgt;
        tgt.out_mode = NTR_OUT_PACKED;
        tgt.packed = r.dst + (size_t)first * r.frame_bytes();
        tgt.aov = aov_offset(aov, (size_t)first * r.frame_pixels(), sc->dev.dim);
        bool p = false;
        if ((rc = enqueue_frame(sc, st, fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, 0, 1, 0, &p,
                                sc->d_views + first, (uint32_t)cnt))) return rc;
    }
    CUDA_TRY(cudaEventRecord(sc->ev1, st));
    sc->timing_valid = true;
    sc->counters = ntr_counters{};
    sc->counters.primary_rays = (uint64_t)n * fmt->width * fmt->height * sc->ss * sc->ss;
    return NTR_OK;
}

NTR_API int ntr_render_views_device(ntr_scene *sc, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                                    void *dev_dst, size_t dst_len, void *stream) {
    ENTER(sc);
    return render_views_device(sc, n, origins, axes, fmt, dev_dst, dst_len, nullptr, stream);
}

NTR_API int ntr_render_views_aovs_device(ntr_scene *sc, int n, const float *origins, const float *axes,
                                         const ntr_image_format *fmt, void *dev_dst, size_t dst_len,
                                         const ntr_aov_buffers *dev_aovs, void *stream) {
    ENTER(sc);
    return render_views_device(sc, n, origins, axes, fmt, dev_dst, dst_len, dev_aovs, stream);
}

NTR_API int ntr_render_float(ntr_scene *sc, int width, int height, float *dst_rgb) {
    ENTER(sc);
    if (width < 1 || height < 1 || !dst_rgb) return fail(NTR_ERR_VALUE, "bad arguments");
    const size_t bytes = (size_t)width * height * 3 * sizeof(float);
    int rc = ensure((void **)&sc->d_accum, &sc->accum_cap, bytes);
    if (rc) return rc;
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_ACCUM;
    tgt.accum = sc->d_accum;
    if ((rc = run_frame_sync(sc, width, height, 0, 0, width, height, nullptr, tgt, 0, 1, 0, sc->stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(dst_rgb, sc->d_accum, bytes, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    return NTR_OK;
}

NTR_API int ntr_calculate_color(ntr_scene *sc, int x, int y, int width, int height, float rgb_out[3]) {
    ENTER(sc);
    if (width < 1 || height < 1 || !rgb_out) return fail(NTR_ERR_VALUE, "bad arguments");
    int rc = ensure((void **)&sc->d_accum, &sc->accum_cap, 3 * sizeof(float));
    if (rc) return rc;
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_ACCUM;
    tgt.accum = sc->d_accum;
    if ((rc = run_frame_sync(sc, width, height, x, y, 1, 1, nullptr, tgt, 0, 1, 0, sc->stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(rgb_out, sc->d_accum, 3 * sizeof(float), cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    return NTR_OK;
}

NTR_API int ntr_primary_hit_ids(ntr_scene *sc, int width, int height, int32_t *ids_out, float *dist_out) {
    ENTER(sc);
    if (width < 1 || height < 1 || !ids_out) return fail(NTR_ERR_VALUE, "bad arguments");
    const size_t n = (size_t)width * height;
    if (sc->ids_cap < n) {
        cudaFree(sc->d_ids); cudaFree(sc->d_dists);
        sc->d_ids = nullptr; sc->d_dists = nullptr; sc->ids_cap = 0;
        CUDA_TRY(cudaMalloc(&sc->d_ids, n * sizeof(int32_t)));
        CUDA_TRY(cudaMalloc(&sc->d_dists, n * sizeof(float)));
        sc->ids_cap = n;
    }
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_IDS;
    tgt.ids = sc->d_ids;
    tgt.dists = sc->d_dists;
    int rc = run_frame_sync(sc, width, height, 0, 0, width, height, nullptr, tgt, 0, 1, 0, sc->stream);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(ids_out, sc->d_ids, n * sizeof(int32_t), cudaMemcpyDeviceToHost, sc->stream));
    if (dist_out) CUDA_TRY(cudaMemcpyAsync(dist_out, sc->d_dists, n * sizeof(float), cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    return NTR_OK;
}

// ---- the camera's rays (ntr_camera_rays) ------------------------------------------------------------------------------
static int check_camera_rays(int width, int height, const float *o, const float *d) {
    if (width < 1 || height < 1 || (uint64_t)width * (uint64_t)height >= (1ull << 31))
        return fail(NTR_ERR_VALUE, "width and height must be at least 1, and width * height below 2^31");
    if (!o || !d) return fail(NTR_ERR_VALUE, "NULL argument");
    return NTR_OK;
}

// Enqueues camera_rays_kernel for the width x height view at factor 1, with the frame parameters enqueue_frame gives it.
static int enqueue_camera_rays(ntr_scene *sc, cudaStream_t st, int width, int height, float *o, float *d) {
    FrameDev f;
    memset(&f, 0, sizeof f);
    f.ss = 1;
    f.width = width; f.height = height;
    f.half_w = (float)width / 2.0f;
    f.half_h = (float)height / 2.0f;
    f.fovI = tanf(sc->dev.fov / 2) / f.half_w;
    f.proj = sc->proj;
    if (sc->proj != NTR_PROJ_PERSPECTIVE) f.proj_k = projection_k(sc->proj, sc->proj_param, f.half_w);
    const uint64_t n = (uint64_t)width * height;
    const int blocks = (int)std::min<uint64_t>((n + kCtaThreads - 1) / kCtaThreads, (uint64_t)sc->sm_count * 16);
    sc->kset(0)->camera_rays(dim3(blocks), dim3(kCtaThreads), st, sc->dev, sc->cam, f, o, d);
    ++sc->launches;
    CUDA_TRY(cudaGetLastError());
    return NTR_OK;
}

NTR_API int ntr_camera_rays(ntr_scene *sc, int width, int height, float *origins_out, float *dirs_out) {
    ENTER(sc);
    int rc = check_camera_rays(width, height, origins_out, dirs_out);
    if (rc) return rc;
    const size_t bytes = (size_t)width * height * sc->dev.dim * sizeof(float), off = align_up(bytes, 256);
    if ((rc = ensure(&sc->d_scratch, &sc->scratch_cap, 2 * off))) return rc;
    float *d_o = static_cast<float *>(sc->d_scratch);
    float *d_d = reinterpret_cast<float *>(static_cast<unsigned char *>(sc->d_scratch) + off);
    if ((rc = enqueue_camera_rays(sc, sc->stream, width, height, d_o, d_d))) return rc;
    CUDA_TRY(cudaMemcpyAsync(origins_out, d_o, bytes, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaMemcpyAsync(dirs_out, d_d, bytes, cudaMemcpyDeviceToHost, sc->stream));
    CUDA_TRY(cudaStreamSynchronize(sc->stream));
    return NTR_OK;
}

NTR_API int ntr_camera_rays_device(ntr_scene *sc, int width, int height, float *origins_out, float *dirs_out, void *stream) {
    ENTER(sc);
    int rc = check_camera_rays(width, height, origins_out, dirs_out);
    if (rc) return rc;
    return enqueue_camera_rays(sc, stream ? (cudaStream_t)stream : sc->stream, width, height, origins_out, dirs_out);
}

static int ray_batch_scratch(ntr_scene *sc, uint32_t n, size_t *offs, const size_t *sizes, int count) {
    size_t total = 0;
    for (int i = 0; i < count; ++i) { offs[i] = total; total += align_up(sizes[i], 256); }
    return ensure(&sc->d_scratch, &sc->scratch_cap, std::max<size_t>(total, 256));
}

NTR_API int ntr_trace_rays_hits(ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, float t_near, float t_far,
                                const uint32_t *skip_ref, const int32_t *skip_lane, int32_t *ids_out, float *dist_out,
                                int32_t *n_transparent_out, int max_hits, int32_t *hit_ids_out, float *hit_dist_out) {
    ENTER(sc);
    if (sc->dev.kind != NTR_SCENE_COMPOSITE) return fail(NTR_ERR_VALUE, "only composite scenes have a k-d tree");
    if (!origins || !dirs || !ids_out) return fail(NTR_ERR_VALUE, "NULL argument");
    if (max_hits < 0 || (max_hits > 0 && !hit_ids_out)) return fail(NTR_ERR_VALUE, "bad transparent-hit output arguments");
    if (n == 0) return NTR_OK;
    const size_t vb = (size_t)n * sc->dev.dim * sizeof(float), ib = (size_t)n * 4, hb = (size_t)n * 4 * (size_t)max_hits;
    size_t offs[9];
    const size_t sizes[9] = {vb, vb, ib, ib, ib, ib, ib, hb, hb};
    int rc = ray_batch_scratch(sc, n, offs, sizes, 9);
    if (rc) return rc;
    unsigned char *b = static_cast<unsigned char *>(sc->d_scratch);
    cudaStream_t st = sc->stream;
    CUDA_TRY(cudaMemcpyAsync(b + offs[0], origins, vb, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b + offs[1], dirs, vb, cudaMemcpyHostToDevice, st));
    if (skip_ref) CUDA_TRY(cudaMemcpyAsync(b + offs[2], skip_ref, ib, cudaMemcpyHostToDevice, st));
    if (skip_lane) CUDA_TRY(cudaMemcpyAsync(b + offs[3], skip_lane, ib, cudaMemcpyHostToDevice, st));
    if (max_hits) CUDA_TRY(cudaMemsetAsync(b + offs[7], 0xFF, hb, st));          // -1: no hit in this slot
    const int flags = sc->base_flags;
    uint32_t ray_blocks = (n + kCtaThreads - 1) / kCtaThreads;
    if (sc->dev.mb_table) ray_blocks = std::min(ray_blocks, sc->dev.mb_threads / kCtaThreads);      // one mailbox column per thread
    sc->kset(flags)->trace_rays(dim3(ray_blocks), dim3(kCtaThreads), st, sc->dev, n,
                                (const float *)(b + offs[0]), (const float *)(b + offs[1]), t_near, t_far,
                                skip_ref ? (const uint32_t *)(b + offs[2]) : nullptr,
                                skip_lane ? (const int32_t *)(b + offs[3]) : nullptr, (int32_t *)(b + offs[4]),
                                (float *)(b + offs[5]), (int32_t *)(b + offs[6]),
                                max_hits ? (int32_t *)(b + offs[7]) : nullptr, max_hits ? (float *)(b + offs[8]) : nullptr, max_hits);
    ++sc->launches;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(ids_out, b + offs[4], ib, cudaMemcpyDeviceToHost, st));
    if (dist_out) CUDA_TRY(cudaMemcpyAsync(dist_out, b + offs[5], ib, cudaMemcpyDeviceToHost, st));
    if (n_transparent_out) CUDA_TRY(cudaMemcpyAsync(n_transparent_out, b + offs[6], ib, cudaMemcpyDeviceToHost, st));
    if (max_hits) {
        CUDA_TRY(cudaMemcpyAsync(hit_ids_out, b + offs[7], hb, cudaMemcpyDeviceToHost, st));
        if (hit_dist_out) CUDA_TRY(cudaMemcpyAsync(hit_dist_out, b + offs[8], hb, cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return NTR_OK;
}

NTR_API int ntr_trace_rays(ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, float t_near, float t_far,
                           const uint32_t *skip_ref, const int32_t *skip_lane, int32_t *ids_out, float *dist_out,
                           int32_t *n_transparent_out) {
    return ntr_trace_rays_hits(sc, n, origins, dirs, t_near, t_far, skip_ref, skip_lane, ids_out, dist_out, n_transparent_out,
                               0, nullptr, nullptr);
}

NTR_API int ntr_occludes_rays(ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, const float *distance,
                              const uint32_t *skip_ref, const int32_t *skip_lane, int32_t *occluded_out,
                              int32_t *n_transparent_out) {
    ENTER(sc);
    if (sc->dev.kind != NTR_SCENE_COMPOSITE) return fail(NTR_ERR_VALUE, "only composite scenes have a k-d tree");
    if (!origins || !dirs || !occluded_out) return fail(NTR_ERR_VALUE, "NULL argument");
    if (n == 0) return NTR_OK;
    const size_t vb = (size_t)n * sc->dev.dim * sizeof(float), ib = (size_t)n * 4;
    size_t offs[7];
    const size_t sizes[7] = {vb, vb, ib, ib, ib, ib, ib};
    int rc = ray_batch_scratch(sc, n, offs, sizes, 7);
    if (rc) return rc;
    unsigned char *b = static_cast<unsigned char *>(sc->d_scratch);
    cudaStream_t st = sc->stream;
    CUDA_TRY(cudaMemcpyAsync(b + offs[0], origins, vb, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(b + offs[1], dirs, vb, cudaMemcpyHostToDevice, st));
    if (distance) CUDA_TRY(cudaMemcpyAsync(b + offs[2], distance, ib, cudaMemcpyHostToDevice, st));
    if (skip_ref) CUDA_TRY(cudaMemcpyAsync(b + offs[3], skip_ref, ib, cudaMemcpyHostToDevice, st));
    if (skip_lane) CUDA_TRY(cudaMemcpyAsync(b + offs[4], skip_lane, ib, cudaMemcpyHostToDevice, st));
    const int flags = sc->base_flags;
    sc->kset(flags)->occludes_rays(dim3((n + kCtaThreads - 1) / kCtaThreads), dim3(kCtaThreads), st, sc->dev, n,
                                   (const float *)(b + offs[0]), (const float *)(b + offs[1]),
                                   distance ? (const float *)(b + offs[2]) : nullptr,
                                   skip_ref ? (const uint32_t *)(b + offs[3]) : nullptr,
                                   skip_lane ? (const int32_t *)(b + offs[4]) : nullptr, (int32_t *)(b + offs[5]),
                                   (int32_t *)(b + offs[6]));
    ++sc->launches;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(occluded_out, b + offs[5], ib, cudaMemcpyDeviceToHost, st));
    if (n_transparent_out) CUDA_TRY(cudaMemcpyAsync(n_transparent_out, b + offs[6], ib, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return NTR_OK;
}


// ---- batches of caller-given rays (ntr_render_rays) ----------------------------------------------------------------------
// A launch covers at most kRaysPerLaunch rays: with two bounce records per ray the wavefront queues then stay at the 2^26
// records a single frame is capped at.  Longer batches run as consecutive launches, each with the regrow-and-retry of a frame.
static const uint32_t kRaysPerLaunch = 1u << 25;

// the AOV buffers of a rays call -> *out (all nullptr for a NULL `aovs`); NTR_ERR_VALUE for a short one
static int check_ray_aovs(uint32_t n, int dim, const ntr_aov_buffers *aovs, AovTarget *out) {
    *out = AovTarget{};
    if (!aovs) return NTR_OK;
    const void *p[3] = {aovs->ids, aovs->depth, aovs->normals};
    const size_t len[3] = {aovs->ids_len, aovs->depth_len, aovs->normals_len}, per[3] = {1, 1, (size_t)dim};
    static const char *const name[3] = {"ids", "depth", "normals"};
    for (int k = 0; k < 3; ++k) {
        if (!p[k]) continue;
        if (len[k] / per[k] < n) return fail(NTR_ERR_VALUE, "the %s buffer is too small for %u rays", name[k], n);
        out->p[k] = const_cast<void *>(p[k]);
    }
    return NTR_OK;
}

static int check_rays(const ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, const float *rgb,
                      const ntr_aov_buffers *aovs, AovTarget *aov) {
    if (n && (!origins || !dirs || !rgb)) return fail(NTR_ERR_VALUE, "NULL argument");
    int rc = check_ray_aovs(n, sc->dev.dim, aovs, aov);
    if (rc) return rc;
    for (const FrameSlot &fs : sc->slots)
        if (fs.open) return fail(NTR_ERR_RUNTIME, "the renderer is already running: a frame of ntr_render_begin is open");
    return NTR_OK;
}

// One scene's share of a rays call, launch after launch.  Host arrays (`host`) go through the scene's scratch memory: the
// rays of a launch are copied in, traced into the scratch accumulator and AOVs, and copied out once the launch needs no
// retry.  Device arrays are read and written in place.
struct RaysRun {
    ntr_scene *sc = nullptr;
    uint32_t n = 0, per = 1, done = 0;
    const float *o = nullptr, *d = nullptr;     // ray 0 of the run
    float *rgb = nullptr;
    AovTarget aov;
    cudaStream_t st = nullptr;
    bool host = false;
    size_t offs[4] = {};                        // scratch: origins, dirs, rgb, AOVs
    FrameJob j{};
    ntr_counters sum{};
};

static int rays_begin(RaysRun &r) {
    ntr_scene *sc = r.sc;
    r.per = std::max<uint32_t>(1, std::min<uint32_t>(sc->rays_per_launch ? sc->rays_per_launch : kRaysPerLaunch, std::max<uint32_t>(r.n, 1)));
    if (!r.host || !r.n) return NTR_OK;
    const size_t vb = (size_t)r.per * sc->dev.dim * sizeof(float);
    const size_t sizes[4] = {vb, vb, (size_t)r.per * 3 * sizeof(float), (size_t)r.per * aov_pixel_bytes(r.aov, sc->dev.dim)};
    return ray_batch_scratch(sc, r.per, r.offs, sizes, 4);
}

static int rays_submit(RaysRun &r) {
    ntr_scene *sc = r.sc;
    const int D = sc->dev.dim;
    const uint32_t cnt = std::min(r.per, r.n - r.done);
    RenderTarget tgt;
    tgt.out_mode = NTR_OUT_RAYS;
    if (r.host) {
        unsigned char *b = static_cast<unsigned char *>(sc->d_scratch);
        const size_t vb = (size_t)cnt * D * sizeof(float);
        CUDA_TRY(cudaMemcpyAsync(b + r.offs[0], r.o + (size_t)r.done * D, vb, cudaMemcpyHostToDevice, r.st));
        CUDA_TRY(cudaMemcpyAsync(b + r.offs[1], r.d + (size_t)r.done * D, vb, cudaMemcpyHostToDevice, r.st));
        tgt.ray_o = (const float *)(b + r.offs[0]);
        tgt.ray_d = (const float *)(b + r.offs[1]);
        tgt.accum = (float *)(b + r.offs[2]);
        tgt.aov = aov_packed(b + r.offs[3], r.aov, cnt, D);
    } else {
        tgt.ray_o = r.o + (size_t)r.done * D;
        tgt.ray_d = r.d + (size_t)r.done * D;
        tgt.accum = r.rgb + (size_t)r.done * 3;
        tgt.aov = aov_offset(r.aov, r.done, D);
    }
    r.j = FrameJob{(int)cnt, 1, 0, 0, (int)cnt, 1, nullptr, tgt, 0, 1, 0, r.st};
    r.j.restart_clock = r.done == 0;
    int rc = frame_submit(sc, r.j);
    if (!rc) rc = frame_readback(sc, r.j);
    return rc;
}

// waits for the launch in flight; once it needs no retry, sums its counters and (host arrays) copies its results out
static int rays_collect(RaysRun &r, bool *again) {
    ntr_scene *sc = r.sc;
    int rc = frame_collect(sc, r.j, again);
    if (rc || *again) return rc;
    add_counters(r.sum, sc->counters);
    r.sum.queue_overflows = sc->counters.queue_overflows;
    const uint32_t cnt = (uint32_t)r.j.win_w;
    if (r.host) {
        const int D = sc->dev.dim;
        CUDA_TRY(cudaMemcpyAsync(r.rgb + (size_t)r.done * 3, r.j.tgt.accum, (size_t)cnt * 3 * sizeof(float), cudaMemcpyDeviceToHost, r.st));
        const AovTarget into = aov_offset(r.aov, r.done, D);
        for (int k = 0; k < 3; ++k)
            if (into.p[k]) CUDA_TRY(cudaMemcpyAsync(into.p[k], r.j.tgt.aov.p[k], (size_t)cnt * aov_bytes(k, D), cudaMemcpyDeviceToHost, r.st));
    }
    r.done += cnt;
    return NTR_OK;
}

// waits for the last copies and publishes the counters
static int rays_finish(RaysRun &r, int rc) {
    const cudaError_t e = cudaStreamSynchronize(r.st);
    if (e != cudaSuccess && !rc) rc = fail(NTR_ERR_RUNTIME, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
    if (!rc) r.sc->counters = r.sum;
    return rc;
}

static int rays_run(RaysRun &r) {
    int rc = rays_begin(r);
    for (int attempt = 0; !rc && r.done < r.n;) {
        if (++attempt > 8) { rc = fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing"); break; }
        bool again = false;
        if (!(rc = rays_submit(r))) rc = rays_collect(r, &again);
        if (!again) attempt = 0;
    }
    return rays_finish(r, rc);
}

NTR_API int ntr_render_rays(ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, float *rgb_out,
                            const ntr_aov_buffers *aovs) {
    ENTER(sc);
    AovTarget aov;
    int rc = check_rays(sc, n, origins, dirs, rgb_out, aovs, &aov);
    if (rc || !n) return rc;
    RaysRun r;
    r.sc = sc; r.n = n; r.o = origins; r.d = dirs; r.rgb = rgb_out; r.aov = aov; r.st = sc->stream; r.host = true;
    return rays_run(r);
}

NTR_API int ntr_render_rays_device(ntr_scene *sc, uint32_t n, const float *origins, const float *dirs, float *rgb_out,
                                   const ntr_aov_buffers *dev_aovs, void *stream) {
    ENTER(sc);
    AovTarget aov;
    int rc = check_rays(sc, n, origins, dirs, rgb_out, dev_aovs, &aov);
    if (rc || !n) return rc;
    RaysRun r;
    r.sc = sc; r.n = n; r.o = origins; r.d = dirs; r.rgb = rgb_out; r.aov = aov;
    r.st = stream ? (cudaStream_t)stream : sc->stream;
    const bool passes = sc->dev.kind == NTR_SCENE_COMPOSITE && sc->any_reflective && sc->dev.max_depth > 0;
    if (passes) return rays_run(r);         // synchronous on the stream, as ntr_render_device with passes
    // single-pass rays: every launch fully asynchronous on the caller's stream
    if ((rc = rays_begin(r))) return rc;
    CUDA_TRY(cudaEventRecord(sc->ev0, r.st));
    for (; r.done < n; r.done += r.per) {
        const uint32_t cnt = std::min(r.per, n - r.done);
        RenderTarget tgt;
        tgt.out_mode = NTR_OUT_RAYS;
        tgt.ray_o = origins + (size_t)r.done * sc->dev.dim;
        tgt.ray_d = dirs + (size_t)r.done * sc->dev.dim;
        tgt.accum = rgb_out + (size_t)r.done * 3;
        tgt.aov = aov_offset(aov, r.done, sc->dev.dim);
        bool p = false;
        if ((rc = enqueue_frame(sc, r.st, (int)cnt, 1, 0, 0, (int)cnt, 1, nullptr, tgt, 0, 1, 0, &p))) return rc;
    }
    CUDA_TRY(cudaEventRecord(sc->ev1, r.st));
    sc->timing_valid = true;
    sc->counters = ntr_counters{};
    sc->counters.primary_rays = n;
    return NTR_OK;
}

NTR_API int ntr_abort(ntr_scene *sc) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    // polled by every warp before it takes the next block of work.  Word 0: a synchronous call in progress, or an
    // asynchronous ntr_render_device frame whose kernels have not finished; words 1..: the open begin/end frames.
    bool async_running = false;
    if (sc->frame_done[0] && !sc->busy.load()) {
        cudaSetDevice(sc->device);
        async_running = cudaEventQuery(sc->frame_done[0]) == cudaErrorNotReady;
        cudaGetLastError();
    }
    if (sc->busy.load() || async_running) sc->h_abort[0] = 1;
    for (int k = 0; k < NTR_FRAMES_IN_FLIGHT; ++k) if (sc->slots[k].open) sc->h_abort[1 + k] = 1;
    return NTR_OK;
}

NTR_API int ntr_get_counters(ntr_scene *sc, ntr_counters *out) {
    if (!sc || !out) return fail(NTR_ERR_VALUE, "NULL argument");
    *out = sc->counters;
    return NTR_OK;
}

NTR_API int ntr_set_instrumented(ntr_scene *sc, int on) {
    if (!sc) return fail(NTR_ERR_VALUE, "scene is NULL");
    sc->instrumented = on != 0;
    return NTR_OK;
}

NTR_API int ntr_last_kernel_ms(ntr_scene *sc, float *ms_out) {
    if (!sc || !ms_out) return fail(NTR_ERR_VALUE, "NULL argument");
    if (!sc->timing_valid) return fail(NTR_ERR_RUNTIME, "nothing has been rendered yet");
    CUDA_TRY(cudaSetDevice(sc->device));
    CUDA_TRY(cudaEventSynchronize(sc->ev1));
    CUDA_TRY(cudaEventElapsedTime(ms_out, sc->ev0, sc->ev1));
    return NTR_OK;
}

NTR_API uint64_t ntr_launch_count(ntr_scene *sc) { return sc ? sc->launches : 0; }

NTR_API int ntr_measure_fp32_peak(int device, float *tflops_out) {
    if (!tflops_out) return fail(NTR_ERR_VALUE, "NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(NTR_ERR_NO_DEVICE, "no CUDA device"); }
    if (device < 0) CUDA_TRY(cudaGetDevice(&device));
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    float *d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 256));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
    fma_peak_kernel<<<blocks, threads>>>(d, 1 << 10);
    float best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        fma_peak_kernel<<<blocks, threads>>>(d, iters);
        cudaEventRecord(e1);
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
        best = std::max(best, (float)(flops / (ms * 1e-3) / 1e12));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops_out = best;
    return NTR_OK;
}

// ---- several GPUs of one box ------------------------------------------------------------------------------------
}  // extern "C"

struct ntr_group {
    std::vector<ntr_scene *> sc;
    std::vector<int> dev;
    unsigned char *d_frame = nullptr;       // on dev[0]; every device stores its tile rows into it (peer access)
    size_t frame_cap = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;           // on dev[0]
    std::vector<cudaEvent_t> done;                      // per device: its part of the frame is complete
    ntr_counters counters{};
    float last_ms = 0;
    bool timing_valid = false;
    std::atomic<bool> busy{false};
};

namespace {

// Traces one frame with every device of the group into g->d_frame.  On return the frame is complete in the memory of
// dev[0] and the stream of sc[0] is ordered behind every device's work (the caller may enqueue a copy on it).
int group_trace(ntr_group *g, const ntr_image_format *fmt) {
    const int n = (int)g->sc.size();
    const size_t bytes = (size_t)fmt->pitch * fmt->height;
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    if (g->frame_cap < bytes) {
        if (g->d_frame) { cudaFree(g->d_frame); g->d_frame = nullptr; g->frame_cap = 0; }
        CUDA_TRY(cudaMalloc(&g->d_frame, bytes + bytes / 8));
        g->frame_cap = bytes + bytes / 8;
    }
    std::vector<FrameJob> jobs(n);
    std::vector<char> pending(n, 1);
    for (int i = 0; i < n; ++i) {
        ntr_scene *sc = g->sc[i];
        if (sc->busy.exchange(true)) {
            for (int k = 0; k < i; ++k) g->sc[k]->busy.store(false);
            return fail(NTR_ERR_RUNTIME, "the renderer is already running");
        }
        sc->h_abort[0] = 0;
        sc->abort_idx = 0;
        RenderTarget tgt;
        tgt.out_mode = NTR_OUT_PACKED;
        tgt.packed = g->d_frame;
        jobs[i] = FrameJob{fmt->width, fmt->height, 0, 0, fmt->width, fmt->height, fmt, tgt, i, n, 0, sc->stream};
    }
    struct Release { ntr_group *g; ~Release() { for (ntr_scene *s : g->sc) s->busy.store(false); } } release{g};
    CUDA_TRY(cudaEventRecord(g->ev0, g->sc[0]->stream));
    int rc = NTR_OK;
    for (int attempt = 0; attempt < 8 && rc == NTR_OK; ++attempt) {
        bool any = false;
        for (int i = 0; i < n && rc == NTR_OK; ++i) {
            if (!pending[i]) continue;
            any = true;
            CUDA_TRY(cudaSetDevice(g->dev[i]));
            if (i && attempt == 0) CUDA_TRY(cudaStreamWaitEvent(g->sc[i]->stream, g->ev0, 0));   // the frame's clock starts on dev[0]
            if ((rc = frame_submit(g->sc[i], jobs[i])) == NTR_OK) rc = frame_readback(g->sc[i], jobs[i]);
        }
        if (!any) break;
        for (int i = 0; i < n; ++i) {
            if (!pending[i]) continue;
            cudaSetDevice(g->dev[i]);
            bool again = false;
            const int r = rc == NTR_OK ? frame_collect(g->sc[i], jobs[i], &again) : (cudaStreamSynchronize(g->sc[i]->stream), NTR_OK);
            if (r != NTR_OK && rc == NTR_OK) rc = r;
            pending[i] = again;
        }
    }
    if (rc == NTR_OK) for (int i = 0; i < n; ++i) if (pending[i]) rc = fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing");
    // order dev[0]'s stream behind the others and stop the frame's clock there
    for (int i = 1; i < n; ++i) {
        cudaSetDevice(g->dev[i]);
        cudaEventRecord(g->done[i], g->sc[i]->stream);
    }
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    for (int i = 1; i < n; ++i) CUDA_TRY(cudaStreamWaitEvent(g->sc[0]->stream, g->done[i], 0));
    CUDA_TRY(cudaEventRecord(g->ev1, g->sc[0]->stream));
    g->timing_valid = rc == NTR_OK;
    if (rc) return rc;
    g->counters = ntr_counters{};
    for (ntr_scene *sc : g->sc) {
        g->counters.primary_rays += sc->counters.primary_rays; g->counters.reflection_rays += sc->counters.reflection_rays;
        g->counters.shadow_rays += sc->counters.shadow_rays; g->counters.node_steps += sc->counters.node_steps;
        g->counters.simplex_tests += sc->counters.simplex_tests; g->counters.solid_tests += sc->counters.solid_tests;
        g->counters.shaded_hits += sc->counters.shaded_hits; g->counters.queue_overflows += sc->counters.queue_overflows;
        g->counters.truncated_hit_lists += sc->counters.truncated_hit_lists;
    }
    return NTR_OK;
}

}  // namespace

extern "C" {

NTR_API int ntr_group_create(const ntr_scene_desc *desc, int n, const int *devices, ntr_group **out) {
    if (!out) return fail(NTR_ERR_VALUE, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(NTR_ERR_NO_DEVICE, "no CUDA device available: ntracer_b200 renders on sm_100a only and has no CPU fallback");
    }
    // a device may be listed more than once: each entry is a chain of passes of its own over its share of the tile rows,
    // and the chains of one device run side by side (one chain's tail beside the other's bulk)
    if (n < 0 || (!devices && n > ndev) || n > 64) return fail(NTR_ERR_VALUE, "the box has %d device(s), %d asked for", ndev, n);
    if (n == 0) n = ndev;
    ntr_group *g = new (std::nothrow) ntr_group();
    if (!g) return fail(NTR_ERR_MEMORY, "out of memory");
    auto bail = [&](int code) { ntr_group_destroy(g); return code; };
    for (int i = 0; i < n; ++i) {
        const int d = devices ? devices[i] : i;
        if (d < 0 || d >= ndev) return bail(fail(NTR_ERR_VALUE, "device %d out of range", d));
        ntr_scene *sc = nullptr;
        const int rc = ntr_scene_create(desc, d, &sc);
        if (rc) return bail(rc);
        g->sc.push_back(sc);
        g->dev.push_back(d);
    }
    // every device stores into the frame buffer of dev[0]
    for (int i = 1; i < n; ++i) {
        int can = 0;
        if (g->dev[i] == g->dev[0]) continue;
        if (cudaDeviceCanAccessPeer(&can, g->dev[i], g->dev[0]) != cudaSuccess || !can)
            return bail(fail(NTR_ERR_RUNTIME, "device %d cannot access the memory of device %d (no peer access)", g->dev[i], g->dev[0]));
        cudaSetDevice(g->dev[i]);
        const cudaError_t e = cudaDeviceEnablePeerAccess(g->dev[0], 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
            return bail(fail(NTR_ERR_RUNTIME, "cudaDeviceEnablePeerAccess failed: %s", cudaGetErrorString(e)));
        cudaGetLastError();
    }
    g->done.assign(n, nullptr);
    for (int i = 0; i < n; ++i) {
        cudaSetDevice(g->dev[i]);
        if (cudaEventCreateWithFlags(&g->done[i], cudaEventDisableTiming) != cudaSuccess) return bail(fail(NTR_ERR_RUNTIME, "cudaEventCreate failed"));
    }
    cudaSetDevice(g->dev[0]);
    if (cudaEventCreate(&g->ev0) != cudaSuccess || cudaEventCreate(&g->ev1) != cudaSuccess) return bail(fail(NTR_ERR_RUNTIME, "cudaEventCreate failed"));
    *out = g;
    return NTR_OK;
}

NTR_API void ntr_group_destroy(ntr_group *g) {
    if (!g) return;
    for (size_t i = 0; i < g->done.size(); ++i) if (g->done[i]) { cudaSetDevice(g->dev[i]); cudaEventDestroy(g->done[i]); }
    if (!g->dev.empty()) {
        cudaSetDevice(g->dev[0]);
        if (!g->sc.empty() && g->sc[0]->stream) cudaStreamSynchronize(g->sc[0]->stream);
        cudaFree(g->d_frame);
        if (g->ev0) cudaEventDestroy(g->ev0);
        if (g->ev1) cudaEventDestroy(g->ev1);
    }
    for (ntr_scene *sc : g->sc) ntr_scene_destroy(sc);
    cudaGetLastError();
    delete g;
}

NTR_API int ntr_group_size(ntr_group *g) { return g ? (int)g->sc.size() : 0; }

NTR_API int ntr_group_set_camera(ntr_group *g, const float *origin, const float *axes) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { const int rc = ntr_scene_set_camera(sc, origin, axes); if (rc) return rc; }
    return NTR_OK;
}

NTR_API int ntr_group_set_params(ntr_group *g, const ntr_scene_desc *desc) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { const int rc = ntr_scene_set_params(sc, desc); if (rc) return rc; }
    return NTR_OK;
}

NTR_API int ntr_group_set_supersampling(ntr_group *g, int factor) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { const int rc = ntr_scene_set_supersampling(sc, factor); if (rc) return rc; }
    return NTR_OK;
}

NTR_API int ntr_group_set_supersampling_threshold(ntr_group *g, float threshold) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { const int rc = ntr_scene_set_supersampling_threshold(sc, threshold); if (rc) return rc; }
    return NTR_OK;
}

NTR_API int ntr_group_set_projection(ntr_group *g, int kind, float param) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { int rc = ntr_scene_set_projection(sc, kind, param); if (rc) return rc; }
    return NTR_OK;
}

NTR_API int ntr_group_last_refine_mask(ntr_group *g, uint8_t *mask, size_t len, uint64_t *count) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    uint64_t total = 0;
    for (ntr_scene *sc : g->sc) {
        uint64_t n = 0;
        const int rc = ntr_last_refine_mask(sc, mask, len, &n);
        if (rc) return rc;
        total += n;
    }
    if (count) *count = total;
    return NTR_OK;
}

NTR_API int ntr_group_render_device(ntr_group *g, const ntr_image_format *fmt, void **dev_frame_out) {
    if (!g || !dev_frame_out) return fail(NTR_ERR_VALUE, "NULL argument");
    int rc = check_format(fmt);
    if (rc) return rc;
    if (g->busy.exchange(true)) return fail(NTR_ERR_RUNTIME, "the renderer is already running");
    rc = group_trace(g, fmt);
    if (rc == NTR_OK && cudaStreamSynchronize(g->sc[0]->stream) != cudaSuccess) rc = fail(NTR_ERR_RUNTIME, "cudaStreamSynchronize failed");
    g->busy.store(false);
    *dev_frame_out = g->d_frame;
    return rc;
}

NTR_API int ntr_group_render(ntr_group *g, const ntr_image_format *fmt, void *dst, size_t dst_len) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    int rc = check_format(fmt);
    if (rc) return rc;
    if (!dst) return fail(NTR_ERR_VALUE, "destination is NULL");
    if (dst_len < (size_t)fmt->pitch * fmt->height) return fail(NTR_ERR_VALUE, "the buffer is too small for an image with the given dimensions");
    if (g->busy.exchange(true)) return fail(NTR_ERR_RUNTIME, "the renderer is already running");
    rc = group_trace(g, fmt);
    if (rc == NTR_OK) {
        // only the pixel bytes are written, like process_pixel: the pitch padding of `dst` is left alone
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (!pinned) {
            rc = download_staged(g->sc[0], static_cast<unsigned char *>(dst), (size_t)fmt->pitch, (size_t)fmt->width * fmt->bytes_per_pixel,
                                 fmt->height, g->d_frame, g->sc[0]->stream);
        } else {
            cudaError_t e = cudaMemcpy2DAsync(dst, (size_t)fmt->pitch, g->d_frame, (size_t)fmt->pitch, (size_t)fmt->width * fmt->bytes_per_pixel,
                                              fmt->height, cudaMemcpyDeviceToHost, g->sc[0]->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(g->sc[0]->stream);
            if (e != cudaSuccess) rc = fail(NTR_ERR_RUNTIME, "device -> host copy failed: %s", cudaGetErrorString(e));
        }
    }
    g->busy.store(false);
    return rc;
}

// Views dealt to the entries in contiguous runs: entry i traces views [i * n / G, (i + 1) * n / G) with the batched kernels
// into its own device memory and copies its frames straight to their place in dst.  Every round submits the next launch on
// every entry before it collects any, so that all devices trace at once.
static int group_render_views(ntr_group *g, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                              void *dst, size_t dst_len, const ntr_aov_buffers *aovs) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) { const int rc = check_views(sc, n, origins, axes, fmt, dst, dst_len); if (rc) return rc; }
    AovTarget aov;
    if (const int rc = check_aovs(n, fmt, g->sc[0]->dev.dim, aovs, &aov)) return rc;
    if (g->busy.exchange(true)) return fail(NTR_ERR_RUNTIME, "the renderer is already running");
    struct Unbusy { ntr_group *g; ~Unbusy() { g->busy.store(false); } } unbusy{g};
    const int G = (int)g->sc.size();
    const size_t fb = (size_t)fmt->pitch * fmt->height;
    unsigned char *const out = static_cast<unsigned char *>(dst);
    int rc = NTR_OK;
    if (frame_adaptive(g->sc[0], NTR_OUT_PACKED)) {
        // adaptive supersampling: view after view through the group's single-view route (ntr_group_render)
        std::vector<CameraDev> saved(G);
        for (int i = 0; i < G; ++i) saved[i] = g->sc[i]->cam;
        ntr_counters sum{};
        for (int k = 0; k < n && !rc; ++k) {
            for (ntr_scene *sc : g->sc) view_camera(sc->cam, origins, axes, sc->dev.dim, k);
            if ((rc = group_trace(g, fmt))) break;
            cudaPointerAttributes attr;
            const bool pinned = cudaPointerGetAttributes(&attr, out) == cudaSuccess && attr.type == cudaMemoryTypeHost;
            cudaGetLastError();
            CUDA_TRY(cudaSetDevice(g->dev[0]));
            if (!pinned) {
                rc = download_staged(g->sc[0], out + k * fb, (size_t)fmt->pitch, (size_t)fmt->width * fmt->bytes_per_pixel,
                                     fmt->height, g->d_frame, g->sc[0]->stream);
            } else {
                CUDA_TRY(cudaMemcpy2DAsync(out + k * fb, (size_t)fmt->pitch, g->d_frame, (size_t)fmt->pitch,
                                           (size_t)fmt->width * fmt->bytes_per_pixel, fmt->height, cudaMemcpyDeviceToHost, g->sc[0]->stream));
                CUDA_TRY(cudaStreamSynchronize(g->sc[0]->stream));
            }
            add_counters(sum, g->counters);
            sum.queue_overflows += g->counters.queue_overflows;
            // the AOVs of the view on the first device (views_aov_pass leaves the frame's refine mask and counters alone)
            if (!rc && aov.any()) rc = views_aovs_of(g->sc[0], origins, axes, k, fmt, aov, false, g->sc[0]->stream);
        }
        for (int i = 0; i < G; ++i) g->sc[i]->cam = saved[i];
        if (!rc) g->counters = sum;
        return rc;
    }
    for (int i = 0; i < G; ++i) {
        ntr_scene *sc = g->sc[i];
        if (sc->busy.exchange(true)) {
            for (int k = 0; k < i; ++k) g->sc[k]->busy.store(false);
            return fail(NTR_ERR_RUNTIME, "the renderer is already running");
        }
        sc->h_abort[0] = 0;
        sc->abort_idx = 0;
    }
    struct Release { ntr_group *g; ~Release() { for (ntr_scene *s : g->sc) s->busy.store(false); } } release{g};
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, dst) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const bool aov_staged = aov.any() && !aovs_pinned(aov);
    std::vector<ViewsRun> runs(G);
    std::vector<int> first(G), attempts(G, 0);
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    CUDA_TRY(cudaEventRecord(g->ev0, g->sc[0]->stream));
    for (int i = 0; i < G && !rc; ++i) {
        ViewsRun &r = runs[i];
        first[i] = (int)((long long)i * n / G);
        r.sc = g->sc[i]; r.fmt = fmt; r.n = (int)((long long)(i + 1) * n / G) - first[i];
        r.dst = out + (size_t)first[i] * fb; r.st = g->sc[i]->stream;
        r.host = true; r.staged = !pinned;
        r.aov = aov_offset(aov, (size_t)first[i] * fmt->width * fmt->height, r.sc->dev.dim); r.aov_staged = aov_staged;
        CUDA_TRY(cudaSetDevice(g->dev[i]));
        if (i) CUDA_TRY(cudaStreamWaitEvent(r.st, g->ev0, 0));      // the call's clock starts on dev[0]
        rc = views_begin(r, origins + (size_t)first[i] * r.sc->dev.dim, axes + (size_t)first[i] * r.sc->dev.dim * r.sc->dev.dim);
    }
    for (bool any = true; any && !rc;) {
        any = false;
        std::vector<char> sent(G, 0);
        for (int i = 0; i < G && !rc; ++i) {
            if (runs[i].done >= runs[i].n) continue;
            if (++attempts[i] > 8) { rc = fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing"); break; }
            cudaSetDevice(g->dev[i]);
            rc = views_submit(runs[i]);
            sent[i] = 1;
            any = true;
        }
        for (int i = 0; i < G; ++i) {
            if (!sent[i]) continue;
            cudaSetDevice(g->dev[i]);
            bool again = false;
            const int r = rc == NTR_OK ? views_collect(runs[i], &again) : (cudaStreamSynchronize(runs[i].st), NTR_OK);
            if (r != NTR_OK && rc == NTR_OK) rc = r;
            if (!again) attempts[i] = 0;
        }
    }
    for (int i = 0; i < G; ++i) {
        cudaSetDevice(g->dev[i]);
        const int r = views_finish(runs[i], rc);
        if (r != NTR_OK && rc == NTR_OK) rc = r;
        if (i) cudaEventRecord(g->done[i], runs[i].st);
    }
    // dev[0]'s stream behind every entry: the call's clock stops when the slowest one is done
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    for (int i = 1; i < G; ++i) CUDA_TRY(cudaStreamWaitEvent(g->sc[0]->stream, g->done[i], 0));
    CUDA_TRY(cudaEventRecord(g->ev1, g->sc[0]->stream));
    g->timing_valid = rc == NTR_OK;
    if (rc) return rc;
    g->counters = ntr_counters{};
    for (const ViewsRun &r : runs) {
        if (r.n < 1) continue;
        add_counters(g->counters, r.sum);
        g->counters.queue_overflows += r.sum.queue_overflows;
    }
    return NTR_OK;
}

NTR_API int ntr_group_render_views(ntr_group *g, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                                   void *dst, size_t dst_len) {
    return group_render_views(g, n, origins, axes, fmt, dst, dst_len, nullptr);
}

NTR_API int ntr_group_render_views_aovs(ntr_group *g, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                                        void *dst, size_t dst_len, const ntr_aov_buffers *aovs) {
    return group_render_views(g, n, origins, axes, fmt, dst, dst_len, aovs);
}

// Rays dealt to the entries in contiguous ranges: entry i traces rays [i * n / G, (i + 1) * n / G) in its own device memory and
// copies its results straight to their place.  Every round submits the next launch on every entry before it collects any.
NTR_API int ntr_group_render_rays(ntr_group *g, uint32_t n, const float *origins, const float *dirs, float *rgb_out,
                                  const ntr_aov_buffers *aovs) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    const int G = (int)g->sc.size();
    AovTarget aov;
    for (ntr_scene *sc : g->sc) { const int rc = check_rays(sc, n, origins, dirs, rgb_out, aovs, &aov); if (rc) return rc; }
    if (!n) return NTR_OK;
    if (g->busy.exchange(true)) return fail(NTR_ERR_RUNTIME, "the renderer is already running");
    struct Unbusy { ntr_group *g; ~Unbusy() { g->busy.store(false); } } unbusy{g};
    for (int i = 0; i < G; ++i) {
        ntr_scene *sc = g->sc[i];
        if (sc->busy.exchange(true)) {
            for (int k = 0; k < i; ++k) g->sc[k]->busy.store(false);
            return fail(NTR_ERR_RUNTIME, "the renderer is already running");
        }
        sc->h_abort[0] = 0;
        sc->abort_idx = 0;
    }
    struct Release { ntr_group *g; ~Release() { for (ntr_scene *s : g->sc) s->busy.store(false); } } release{g};
    const int D = g->sc[0]->dev.dim;
    std::vector<RaysRun> runs(G);
    std::vector<int> attempts(G, 0);
    int rc = NTR_OK;
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    CUDA_TRY(cudaEventRecord(g->ev0, g->sc[0]->stream));
    for (int i = 0; i < G && !rc; ++i) {
        RaysRun &r = runs[i];
        const uint32_t first = (uint32_t)((uint64_t)i * n / G);
        r.sc = g->sc[i]; r.n = (uint32_t)((uint64_t)(i + 1) * n / G) - first;
        r.o = origins + (size_t)first * D; r.d = dirs + (size_t)first * D; r.rgb = rgb_out + (size_t)first * 3;
        r.aov = aov_offset(aov, first, D); r.st = g->sc[i]->stream; r.host = true;
        CUDA_TRY(cudaSetDevice(g->dev[i]));
        if (i) CUDA_TRY(cudaStreamWaitEvent(r.st, g->ev0, 0));      // the call's clock starts on dev[0]
        rc = rays_begin(r);
    }
    for (bool any = true; any && !rc;) {
        any = false;
        std::vector<char> sent(G, 0);
        for (int i = 0; i < G && !rc; ++i) {
            if (runs[i].done >= runs[i].n) continue;
            if (++attempts[i] > 8) { rc = fail(NTR_ERR_RUNTIME, "wavefront queue kept overflowing"); break; }
            cudaSetDevice(g->dev[i]);
            rc = rays_submit(runs[i]);
            sent[i] = 1;
            any = true;
        }
        for (int i = 0; i < G; ++i) {
            if (!sent[i]) continue;
            cudaSetDevice(g->dev[i]);
            bool again = false;
            const int r = rc == NTR_OK ? rays_collect(runs[i], &again) : (cudaStreamSynchronize(runs[i].st), NTR_OK);
            if (r != NTR_OK && rc == NTR_OK) rc = r;
            if (!again) attempts[i] = 0;
        }
    }
    for (int i = 0; i < G; ++i) {
        cudaSetDevice(g->dev[i]);
        const int r = rays_finish(runs[i], rc);
        if (r != NTR_OK && rc == NTR_OK) rc = r;
        if (i) cudaEventRecord(g->done[i], runs[i].st);
    }
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    for (int i = 1; i < G; ++i) CUDA_TRY(cudaStreamWaitEvent(g->sc[0]->stream, g->done[i], 0));
    CUDA_TRY(cudaEventRecord(g->ev1, g->sc[0]->stream));
    g->timing_valid = rc == NTR_OK;
    if (rc) return rc;
    g->counters = ntr_counters{};
    for (const RaysRun &r : runs) {
        add_counters(g->counters, r.sum);
        g->counters.queue_overflows += r.sum.queue_overflows;
    }
    return NTR_OK;
}

NTR_API int ntr_group_abort(ntr_group *g) {
    if (!g) return fail(NTR_ERR_VALUE, "group is NULL");
    for (ntr_scene *sc : g->sc) ntr_abort(sc);
    return NTR_OK;
}

NTR_API int ntr_group_get_counters(ntr_group *g, ntr_counters *out) {
    if (!g || !out) return fail(NTR_ERR_VALUE, "NULL argument");
    *out = g->counters;
    return NTR_OK;
}

NTR_API int ntr_group_last_kernel_ms(ntr_group *g, float *ms_out) {
    if (!g || !ms_out) return fail(NTR_ERR_VALUE, "NULL argument");
    if (!g->timing_valid) return fail(NTR_ERR_RUNTIME, "nothing has been rendered yet");
    CUDA_TRY(cudaSetDevice(g->dev[0]));
    CUDA_TRY(cudaEventSynchronize(g->ev1));
    CUDA_TRY(cudaEventElapsedTime(ms_out, g->ev0, g->ev1));
    return NTR_OK;
}

NTR_API uint64_t ntr_group_launch_count(ntr_group *g) {
    uint64_t n = 0;
    if (g) for (ntr_scene *sc : g->sc) n += sc->launches;
    return n;
}

// ---- frame buffers shared between processes (one process per GPU) ----------------------------------------------
NTR_API int ntr_frame_alloc(int device, size_t bytes, void **dev_ptr_out) {
    if (!dev_ptr_out || !bytes) return fail(NTR_ERR_VALUE, "bad arguments");
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMalloc(dev_ptr_out, bytes));       // a dedicated allocation: its base address is what cudaIpcGetMemHandle exports
    return NTR_OK;
}
NTR_API int ntr_frame_free(int device, void *dev_ptr) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaFree(dev_ptr));
    return NTR_OK;
}
NTR_API int ntr_frame_export(void *dev_ptr, unsigned char handle_out[NTR_IPC_HANDLE_BYTES]) {
    static_assert(sizeof(cudaIpcMemHandle_t) <= NTR_IPC_HANDLE_BYTES, "IPC handle size");
    if (!dev_ptr || !handle_out) return fail(NTR_ERR_VALUE, "NULL argument");
    cudaIpcMemHandle_t h;
    CUDA_TRY(cudaIpcGetMemHandle(&h, dev_ptr));
    memset(handle_out, 0, NTR_IPC_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof h);
    return NTR_OK;
}
NTR_API int ntr_frame_import(int device, const unsigned char handle[NTR_IPC_HANDLE_BYTES], void **dev_ptr_out) {
    if (!handle || !dev_ptr_out) return fail(NTR_ERR_VALUE, "NULL argument");
    CUDA_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return NTR_OK;
}
NTR_API int ntr_frame_release(int device, void *imported_ptr) {
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaIpcCloseMemHandle(imported_ptr));
    return NTR_OK;
}
NTR_API int ntr_frame_fill(int device, void *dev_ptr, int value, size_t bytes, void *stream) {
    if (!dev_ptr) return fail(NTR_ERR_VALUE, "NULL argument");
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMemsetAsync(dev_ptr, value, bytes, (cudaStream_t)stream));
    return NTR_OK;
}
NTR_API int ntr_frame_download(int device, const void *dev_ptr, const ntr_image_format *fmt, void *dst, size_t dst_len, void *stream) {
    int rc = check_format(fmt);
    if (rc) return rc;
    if (!dev_ptr || !dst) return fail(NTR_ERR_VALUE, "NULL argument");
    if (dst_len < (size_t)fmt->pitch * fmt->height) return fail(NTR_ERR_VALUE, "the buffer is too small for an image with the given dimensions");
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaMemcpy2DAsync(dst, (size_t)fmt->pitch, dev_ptr, (size_t)fmt->pitch, (size_t)fmt->width * fmt->bytes_per_pixel, fmt->height,
                               cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return NTR_OK;
}

}  // extern "C"
