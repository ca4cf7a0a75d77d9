/* ntracer_b200 -- C ABI of the B200 (sm_100a) backend for NTracer's per-pixel render loop.
 *
 * This is the drop-in boundary (DESIGN.md section 2, SURVEY.md section 8b).  It sits exactly where the
 * reference crosses from its Python type objects into `scene::calculate_color` / `worker_draw`:
 * plain pointers and sizes, no C++/torch/Python types, never throws.  Every entry point cites the
 * reference interface it replaces (paths are relative to the reference tree, /root/reference).
 * INTEGRATION.md shows the binding a maintainer adds to src/render.cpp / src/ntracer_body.hpp.
 *
 * Conventions
 *   - every function returns NTR_OK (0) or a negative ntr_status; ntr_last_error() returns a
 *     thread-local, NUL-terminated description of the last failure on the calling thread
 *     (the reference converts C++ exceptions to Python ones in PY_EXCEPT_HANDLERS,
 *     src/py_common.hpp:39-47: bad_alloc -> MemoryError, std::exception -> RuntimeError,
 *     ValueError for bad formats/buffers -- the status codes below keep that split);
 *   - all arithmetic is FP32 (`real` = float, src/geometry.hpp:11);
 *   - "D" below is the scene dimension (3..NTR_MAX_DIM).
 */
#ifndef NTRACER_B200_H
#define NTRACER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define NTR_API
#else
#define NTR_API __attribute__((visibility("default")))
#endif

#define NTR_ABI_VERSION 1
#define NTR_MAX_DIM 16          /* runtime-dimension kernels keep vectors of this many floats */
#define NTR_MAX_CHANNELS 16     /* MAX_PIXELSIZE = 16 bytes, src/render.cpp:50 */
#define NTR_MAX_TREE_DEPTH 62   /* traversal stack entries (reference default max depth 25, src/tracer.hpp:41) */

typedef enum ntr_status {
    NTR_OK = 0,
    NTR_ERR_VALUE = -1,         /* ValueError: bad argument / format / buffer size            */
    NTR_ERR_MEMORY = -2,        /* MemoryError: host or device allocation failed               */
    NTR_ERR_RUNTIME = -3,       /* RuntimeError: CUDA failure, "the renderer is already running" */
    NTR_ERR_NO_DEVICE = -4,     /* no CUDA device / kernels not built for it: there is NO CPU fallback */
    NTR_ERR_ABORTED = -5        /* render was aborted (BlockingRenderer.render returns False)   */
} ntr_status;

enum { NTR_SCENE_BOX = 0, NTR_SCENE_COMPOSITE = 1 };       /* box_scene / composite_scene, src/tracer.hpp:83,1710 */
enum { NTR_SOLID_CUBE = 1, NTR_SOLID_SPHERE = 2 };         /* enum solid_type, src/tracer.hpp:225 */

#define NTR_NULL_NODE 0xFFFFFFFFu     /* null child pointer of kd_branch (src/tracer.hpp:816-817) */
#define NTR_LEAF_FLAG 0x80000000u
#define NTR_REF_SIMPLEX 0u            /* leaf_refs[i] = (type << 30) | index */
#define NTR_REF_BATCH 1u              /* index = first of `batch_size` consecutive simplex records (triangle_batch lanes) */
#define NTR_REF_SOLID 2u

/* 16-byte k-d tree node.  Replaces kd_branch{axis,split,left,right} and kd_leaf{size,batches,items}
 * (src/tracer.hpp:813-830, 836-856, 950-975).
 *   branch: meta = axis,                     w1 = float bits of split, w2 = left node, w3 = right node
 *   leaf:   meta = NTR_LEAF_FLAG | n_batches, w1 = first index into leaf_refs, w2 = item count, w3 = 0 */
typedef struct ntr_node {
    uint32_t meta, w1, w2, w3;
} ntr_node;

/* Scene description handed to ntr_scene_create.  Everything is copied (into the device arena);
 * the caller's arrays may be freed afterwards.  This is what `geom_allocator` uploads in the
 * north-star design; in the reference the same data lives in Python-owned heap objects reachable
 * from composite_scene::root (src/tracer.hpp:1713-1725). */
typedef struct ntr_scene_desc {
    int32_t dim;                    /* D */
    int32_t kind;                   /* NTR_SCENE_BOX | NTR_SCENE_COMPOSITE */
    int32_t batch_size;             /* v_real::size of the tree's triangle_batch items (1 if none) */
    uint32_t root;                  /* index of the root node, NTR_NULL_NODE for an empty tree */
    uint32_t n_nodes;
    const ntr_node *nodes;
    uint32_t n_leaf_refs;
    const uint32_t *leaf_refs;
    uint32_t n_simplex;
    const float *simplex;           /* n_simplex x ((D+1)*D+1): face_normal[D], d, p1[D], edge_normals[D-1][D]
                                       (triangle / triangle_batch members, src/tracer.hpp:392-401,539-541) */
    const int32_t *simplex_mat;     /* material index per simplex (per batch lane, src/tracer.hpp:209) */
    uint32_t n_solids;
    const float *solids;            /* n_solids x (1+2*D*D+D): type, orientation[D*D], inv_orientation[D*D],
                                       position[D]  (struct solid, src/tracer.hpp:231-249) */
    const int32_t *solid_mat;
    uint32_t n_materials;
    const float *materials;         /* n_materials x 10: color[3], specular[3], opacity, reflectivity,
                                       specular_intensity, specular_exp  (struct material, src/render.hpp:56-73) */
    const float *boundary;          /* 2 x D: aabb start, end (composite_scene::boundary) */
    /* composite_scene state, defaults src/tracer.hpp:1727-1740 */
    float fov;
    int32_t shadows;
    int32_t camera_light;
    int32_t max_reflect_depth;      /* 0..63 (one wavefront pass per depth; more is NTR_ERR_VALUE) */
    int32_t bg_gradient_axis;
    float ambient[3], bg1[3], bg2[3], bg3[3];
    uint32_t n_point_lights;
    const float *point_lights;      /* n x (D+3): position[D], color[3]   (point_light, src/tracer.hpp:1678-1689) */
    uint32_t n_global_lights;
    const float *global_lights;     /* n x (D+3): direction[D], color[3]  (global_light, src/tracer.hpp:1691-1698) */
} ntr_scene_desc;

/* struct channel / struct image_format, src/render.cpp:95-99,167-172 */
typedef struct ntr_channel {
    float f_r, f_g, f_b, f_c;
    uint8_t bit_size;               /* 1..31, or 32 when tfloat */
    uint8_t tfloat;
    uint8_t pad_[2];
} ntr_channel;

typedef struct ntr_image_format {
    int32_t width, height, pitch;   /* pitch in bytes, >= width*bytes_per_pixel */
    int32_t n_channels;
    ntr_channel channels[NTR_MAX_CHANNELS];
    uint8_t bytes_per_pixel;        /* ceil(sum(bit_size)/8), <= 16 */
    uint8_t reversed;
    uint8_t pad_[2];
} ntr_image_format;

/* Ray / work counters of the last render (SURVEY.md section 8d "ray counting"). */
typedef struct ntr_counters {
    uint64_t primary_rays;          /* W*H, times s*s for a supersampling factor s (ntr_scene_set_supersampling) */
    uint64_t reflection_rays;       /* recursive ray_color calls, src/tracer.hpp:1843 */
    uint64_t shadow_rays;           /* light_reaches calls, src/tracer.hpp:1787,1811 */
    uint64_t node_steps;            /* kd_branch visits (only filled by instrumented renders) */
    uint64_t simplex_tests;         /* simplex tests, every batch lane counted (instrumented renders) */
    uint64_t solid_tests;
    uint64_t shaded_hits;           /* base_color calls */
    uint64_t queue_overflows;       /* wavefront queue regrow events */
    uint64_t truncated_hit_lists;   /* rays whose list of transparent hits outgrew the 16 entries the kernels keep (the
                                       reference preallocates 10 and is undefined beyond, src/tracer.hpp:26,670-680):
                                       their farthest layers are missing from the frame -- 0 means nothing was cut */
} ntr_counters;

typedef struct ntr_scene ntr_scene;     /* opaque: device arena + streams + queues of one scene on one GPU */

/* ---- library / device ------------------------------------------------------------------------ */
NTR_API int ntr_abi_version(void);
NTR_API const char *ntr_last_error(void);
/* Number of usable sm_100 devices (0 when there is none: every compute call then fails with
 * NTR_ERR_NO_DEVICE -- there is no CPU path in this library). */
NTR_API int ntr_device_count(void);

/* ---- scene lifetime: replaces composite_scene / box_scene construction + geom_allocator ------- */
/* device < 0: use the current CUDA device. */
NTR_API int ntr_scene_create(const ntr_scene_desc *desc, int device, ntr_scene **out);
NTR_API void ntr_scene_destroy(ntr_scene *scene);
/* camera<Store>{origin, t_orientation} (src/camera.hpp:7-46): origin[D], axes[D*D] row-major;
 * rows 0,1,2 = right, up, forward.  Replaces Scene.set_camera (src/ntracer_body.hpp:833-844). */
NTR_API int ntr_scene_set_camera(ntr_scene *scene, const float *origin, const float *axes);
/* Re-sends the mutable composite_scene state of `desc` (fov, shadows, camera_light, max_reflect_depth,
 * background, ambient, lights) without touching geometry.  Replaces the set_* mutators
 * (src/ntracer_body.hpp:833-933). */
NTR_API int ntr_scene_set_params(ntr_scene *scene, const ntr_scene_desc *desc);
/* Supersampled anti-aliasing (no counterpart in the reference, which traces one ray through the corner of every pixel).
 * factor s in 1..NTR_MAX_SUPERSAMPLING, default 1; anything else -> NTR_ERR_VALUE.  Host state like the camera: read when
 * a frame is enqueued (ntr_render_begin captures it with the camera).  s = 1 is the plain renderer, byte for byte.
 * With s > 1 the float colour of output pixel (x, y) of a W x H frame is the box-filtered mean of the s x s pixels
 * (s*x + i, s*y + j) of the sW x sH view, summed j-major, i-minor: each sample's colour is computed exactly as
 * ntr_render_float(sW, sH) computes that pixel, with every contribution weighted by 1/(s*s), and added to the pixel's sum;
 * the sum is then packed as usual (the mean is taken before clamping).  For s in {2, 4, 8} and frames without reflections
 * the result is bit-identical to that mean of the big view.  ntr_render, ntr_render_device, ntr_render_begin/end,
 * ntr_render_float, ntr_calculate_color and ntr_group_render* honour it; ntr_primary_hit_ids, ntr_trace_rays* and
 * ntr_occludes_rays are per-ray hooks and ignore it.  Counters: primary_rays = s*s per pixel, the others are those of the
 * big view.  The wavefront queues of reflective scenes hold up to s*s times the bounces of a plain frame: their memory
 * grows with s*s (see README). */
#define NTR_MAX_SUPERSAMPLING 8
NTR_API int ntr_scene_set_supersampling(ntr_scene *scene, int factor);
/* Adaptive supersampling: trace the s x s samples only where a pixel's corner colours disagree.  threshold t < 0 (the
 * default) is off: the full supersampling above, byte for byte; NaN or +inf -> NTR_ERR_VALUE.  Host state like the factor,
 * ignored at factor 1 (the same kernels and launches as without it).  With s > 1 and t >= 0, c(x, y) is the plain 1-spp
 * float colour of view pixel (x, y) (what factor 1 gives); pixel (x, y) is refined iff, for some channel k,
 * max c_k(p) - min c_k(p) > t over p in {(x, y), (x+1, y), (x, y+1), (x+1, y+1)} intersected with the VIEW (float32, RGB,
 * before packing).  A refined pixel's float colour is that of full supersampling at factor s, any other pixel's is c(x, y);
 * then the frame is packed as usual.  Without reflection passes both parts are bit-identical to the full-SS and the plain
 * frame; with them every pixel stays within 1 LSB, and the mask may differ where a pixel's contrast lies within float
 * rounding of t (the bounce passes add with float atomics).  Counters: primary_rays = traced plain pixels (the window's own
 * pixels and the halo of corner pixels a sharded render or a calculate_color window needs beyond them) + refined pixels *
 * s*s; the others are summed over everything traced.  Every path that honours the factor honours the threshold
 * (ntr_render_begin captures it with the camera); the per-ray hooks ignore it.  Adaptive frames are traced synchronously
 * like frames with reflection passes. */
NTR_API int ntr_scene_set_supersampling_threshold(ntr_scene *scene, float threshold);
/* The refine mask of the last completed frame: one byte (1 = refined) per pixel of its window, row-major with a row of
 * the window's width (for ntr_calculate_color: 1 x 1); len must cover the window or NTR_ERR_VALUE.  A sharded render
 * (tile-row interleave) writes only its own rows.  *count_or_null receives the number of refined pixels.  A frame that
 * was not adaptively supersampled has an all-zero mask.  NTR_ERR_RUNTIME before the first frame.  Either pointer may be
 * NULL. */
NTR_API int ntr_last_refine_mask(ntr_scene *scene, uint8_t *mask_or_null, size_t len, uint64_t *count_or_null);

/* ---- the hot path ---------------------------------------------------------------------------- */
/* Renders one frame into a HOST buffer: replaces worker_draw + process_pixel for all tiles
 * (src/render.cpp:396-493) as driven by BlockingRenderer.render (src/render.cpp:853-909).
 * dst_len must be >= pitch*height (im_check_buffer_size, src/render.cpp:187-190).
 * Returns NTR_ERR_ABORTED if ntr_abort() was called while it ran. */
NTR_API int ntr_render(ntr_scene *scene, const ntr_image_format *fmt, void *dst, size_t dst_len);
/* Same, into DEVICE memory on a caller-supplied CUDA stream (cudaStream_t passed as void*; NULL =
 * the scene's own stream), asynchronously.  Only the tile rows ty with
 * ty % tile_row_step == tile_row_first are rendered (32-pixel rows, RENDER_CHUNK_SIZE,
 * src/render.cpp:43); the others are left untouched.  If `compact` is non-zero the rendered tile
 * rows are stored back to back (tile row k of this rank at byte offset k*32*pitch) -- the layout
 * the multi-GPU gather uses; otherwise at their frame position. */
NTR_API int ntr_render_device(ntr_scene *scene, const ntr_image_format *fmt, void *dev_dst, size_t dst_len,
                              void *stream, int tile_row_first, int tile_row_step, int compact);
/* The interactive loop (SURVEY 8(f)-3): CallbackRenderer.begin_render + completion (src/render.cpp:495-563,
 * 651-700) as driven by scripts/polytope.py:505-557 (rotating camera, one frame after the other).
 * ntr_render_begin enqueues the frame with the camera / parameters current at the call and returns a ticket
 * without waiting; ntr_render_end(ticket) waits for that frame and completes the copy into the `dst` given
 * to begin.  Up to NTR_FRAMES_IN_FLIGHT frames may be open: frame k+1 is traced while frame k crosses PCIe
 * (double-buffered device frames + pinned staging; `dst` is written directly when it is itself pinned).
 * The camera may be changed between begin and end (it is captured at begin).  `dst` must stay valid until end.
 * Tickets must be ended in the order they were begun.  A third begin without an end -> NTR_ERR_RUNTIME
 * ("already running", src/render.cpp:676).  ntr_render_end returns NTR_ERR_ABORTED if ntr_abort() hit the frame. */
#define NTR_FRAMES_IN_FLIGHT 2
NTR_API int ntr_render_begin(ntr_scene *scene, const ntr_image_format *fmt, void *dst, size_t dst_len,
                             uint64_t *ticket_out);
NTR_API int ntr_render_end(ntr_scene *scene, uint64_t ticket);
/* A batch of camera views in one call (no counterpart in the reference): origins is n x D and axes n x D x D, each view in
 * the layout of ntr_scene_set_camera.  Frame k is written at byte offset k*pitch*height of dst (dst_len must be at least
 * n*pitch*height); only pixel bytes are written, the pitch padding is left alone.  Frame k is what ntr_render produces after
 * ntr_scene_set_camera(origins[k], axes[k]) with the scene's current parameters and supersampling factor: byte-identical
 * for frames without reflection passes (BoxScenes and every factor, 1 included), within 1 LSB per channel with them
 * (float atomics add in no fixed order).  The scene's own camera is unchanged afterwards.
 * The views share launches: one persistent launch per pass covers up to V views (V*width*height*factor^2 <= 2^25; the
 * environment variable NTR_VIEWS_PER_LAUNCH=V overrides), so each bounce depth of all views is one pass, and the frames of
 * one launch cross PCIe while the next is traced.  Counters are the sums over the views (primary_rays =
 * n*width*height*factor^2).  With a supersampling threshold set (adaptive supersampling) the views are rendered one after
 * the other through the ntr_render route instead, and ntr_last_refine_mask describes the last view.
 * NTR_ERR_VALUE: n < 1, a NULL pointer, a bad format or a short buffer.  NTR_ERR_RUNTIME while a frame of the scene is
 * rendering or open (ntr_render_begin).  NTR_ERR_ABORTED after ntr_abort(); the frames' contents are then unspecified. */
NTR_API int ntr_render_views(ntr_scene *scene, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                             void *dst, size_t dst_len);
/* The same frames into DEVICE memory of the scene's device, on a caller-supplied CUDA stream (NULL = the scene's own):
 * asynchronous when the frames need a single pass, synchronous on that stream with reflection passes, as ntr_render_device. */
NTR_API int ntr_render_views_device(ntr_scene *scene, int n, const float *origins, const float *axes,
                                    const ntr_image_format *fmt, void *dev_dst, size_t dst_len, void *stream);
/* Per-pixel auxiliary outputs (AOVs) of a views call (no counterpart in the reference).  For view k and output pixel (x, y),
 * at index (k*height + y)*width + x, they describe the pixel's plain primary ray -- the factor-1 ray ntr_primary_hit_ids
 * traces after ntr_scene_set_camera(origins[k], axes[k]) -- whatever the supersampling factor or threshold:
 *   ids      the flat id of its opaque hit as ntr_primary_hit_ids defines it (-1: a miss; transparent layers are not hits),
 *   depth    its distance along the ray (0 on a miss), both bit-identical to ntr_primary_hit_ids,
 *   normals  dim floats per pixel: the normal that shades the hit (RayIntersection.normal of the reference: a simplex's unit
 *            face normal facing the ray, a solid's back-transformed normal as it is, a BoxScene face's axis vector), zeros
 *            on a miss.
 * A NULL pointer means "not wanted"; each *_len counts elements (n*width*height, times dim for the normals). */
typedef struct ntr_aov_buffers {
    int32_t *ids;
    float *depth;
    float *normals;
    size_t ids_len, depth_len, normals_len;
} ntr_aov_buffers;
/* ntr_render_views plus the AOVs in the same launches, into host memory; the frames and counters are those of ntr_render_views
 * (the rays traced for the AOVs are not counted).  aovs == NULL or all three NULL is ntr_render_views.  A launch then covers
 * at most as many views as keep its AOVs within about 1 GB (NTR_VIEWS_PER_LAUNCH still overrides).  NTR_ERR_VALUE also for
 * a short AOV buffer, checked before any work; after NTR_ERR_ABORTED the AOVs' contents are unspecified. */
NTR_API int ntr_render_views_aovs(ntr_scene *scene, int n, const float *origins, const float *axes, const ntr_image_format *fmt,
                                  void *dst, size_t dst_len, const ntr_aov_buffers *aovs);
/* The same with the frames and the AOVs in DEVICE memory of the scene's device, on a caller-supplied stream, as
 * ntr_render_views_device. */
NTR_API int ntr_render_views_aovs_device(ntr_scene *scene, int n, const float *origins, const float *axes,
                                         const ntr_image_format *fmt, void *dev_dst, size_t dst_len,
                                         const ntr_aov_buffers *dev_aovs, void *stream);
/* Float RGB of every pixel (3 floats per pixel, row-major) = scene::calculate_color for the whole
 * view (src/render.hpp:12-13) before channel packing; host destination. */
NTR_API int ntr_render_float(ntr_scene *scene, int width, int height, float *dst_rgb);
/* Scene.calculate_color(x,y,width,height) (src/render.cpp:586-614). */
NTR_API int ntr_calculate_color(ntr_scene *scene, int x, int y, int width, int height, float rgb_out[3]);
/* Primary-ray hit ids: for every pixel the flat primitive id of the opaque hit of
 * intersects(root, primary ray) (src/tracer.hpp:1245-1256,1863) or -1.  Flat id = simplex index
 * (batch lanes are consecutive records), solids follow at n_simplex + solid index.
 * dist_out (optional) receives the hit distance (0 on miss). */
NTR_API int ntr_primary_hit_ids(ntr_scene *scene, int width, int height, int32_t *ids_out, float *dist_out);
/* KDNode.intersects / KDNode.occludes for a batch of arbitrary rays (src/ntracer_body.hpp:1412-1496):
 * origins/dirs are n x D.  skip_ref / skip_lane: per-ray `source` primitive as a leaf_refs value and
 * batch lane (NULL = none).  ids_out: flat id of the opaque hit or -1; dist_out: its distance;
 * n_transparent_out (optional): number of transparent hits that survived trimming. */
NTR_API int ntr_trace_rays(ntr_scene *scene, uint32_t n, const float *origins, const float *dirs,
                           float t_near, float t_far, const uint32_t *skip_ref, const int32_t *skip_lane,
                           int32_t *ids_out, float *dist_out, int32_t *n_transparent_out);
/* The same with the transparent hits themselves: KDNode.intersects returns every surviving transparent hit as a
 * RayIntersection ahead of the opaque one (src/ntracer_body.hpp:1438-1456, 1759-1766).  hit_ids_out / hit_dist_out are
 * n x max_hits: flat primitive id (-1 = unused slot) and distance of the first max_hits entries of the ray's list, in
 * the list's order (unsorted, as the reference's quick_list leaves them after trimming; the kernels keep up to 16). */
NTR_API int ntr_trace_rays_hits(ntr_scene *scene, uint32_t n, const float *origins, const float *dirs,
                                float t_near, float t_far, const uint32_t *skip_ref, const int32_t *skip_lane,
                                int32_t *ids_out, float *dist_out, int32_t *n_transparent_out, int max_hits,
                                int32_t *hit_ids_out, float *hit_dist_out);
NTR_API int ntr_occludes_rays(ntr_scene *scene, uint32_t n, const float *origins, const float *dirs,
                              const float *distance, const uint32_t *skip_ref, const int32_t *skip_lane,
                              int32_t *occluded_out, int32_t *n_transparent_out);

/* ---- several GPUs of one box (SURVEY.md section 8e; no counterpart in the reference, whose parallelism is worker
 * threads pulling 32x32 tiles, src/render.cpp:468-493,829-838) ---------------------------------------------------
 * A group replicates the scene on n devices.  A frame is split by interleaved 32-pixel tile rows (tile row ty belongs
 * to device ty % n, which balances the centre-heavy cost of polytope scenes); every device traces its rows and its
 * packing epilogue stores the pixels straight into ONE frame buffer in the memory of the first device, over NVLink
 * (peer access) -- there is no gather step and no second copy; one device->host transfer follows.  This is what
 * BlockingRenderer(threads=N) maps to ("threads" = how many workers trace the frame).
 * devices = NULL: the first n usable devices.  n = 0: all of them.  Every device must be able to reach devices[0]. */
typedef struct ntr_group ntr_group;
NTR_API int ntr_group_create(const ntr_scene_desc *desc, int n, const int *devices, ntr_group **out);
NTR_API void ntr_group_destroy(ntr_group *group);
NTR_API int ntr_group_size(ntr_group *group);
NTR_API int ntr_group_set_camera(ntr_group *group, const float *origin, const float *axes);
NTR_API int ntr_group_set_params(ntr_group *group, const ntr_scene_desc *desc);
/* ntr_scene_set_supersampling for every device of the group. */
NTR_API int ntr_group_set_supersampling(ntr_group *group, int factor);
/* ntr_scene_set_supersampling_threshold for every device of the group. */
NTR_API int ntr_group_set_supersampling_threshold(ntr_group *group, float threshold);
/* ntr_last_refine_mask of the last group frame: every device writes its tile rows, the count is their sum. */
NTR_API int ntr_group_last_refine_mask(ntr_group *group, uint8_t *mask_or_null, size_t len, uint64_t *count_or_null);
/* ntr_render over the group: host destination, same contract (NTR_ERR_ABORTED after ntr_group_abort). */
NTR_API int ntr_group_render(ntr_group *group, const ntr_image_format *fmt, void *dst, size_t dst_len);
/* The same frame left in device memory: *dev_frame_out receives the frame buffer on the first device (pitch*height
 * bytes, owned by the group, valid until the next render of the group). */
NTR_API int ntr_group_render_device(ntr_group *group, const ntr_image_format *fmt, void **dev_frame_out);
/* ntr_render_views over the group, whole views per device: entry i (a device listed twice is two entries) gets views
 * [floor(i*n/G), floor((i+1)*n/G)), traces them with the batched kernels into its own memory and copies its frames straight
 * to their place in dst; no frame is split and nothing crosses NVLink.  Counters are summed over the entries,
 * ntr_group_last_kernel_ms is the slowest entry's.  With a supersampling threshold set, view after view via ntr_group_render. */
NTR_API int ntr_group_render_views(ntr_group *group, int n, const float *origins, const float *axes,
                                   const ntr_image_format *fmt, void *dst, size_t dst_len);
/* ntr_render_views_aovs over the group: every entry writes the frames and AOVs of its own views straight to their place. */
NTR_API int ntr_group_render_views_aovs(ntr_group *group, int n, const float *origins, const float *axes,
                                        const ntr_image_format *fmt, void *dst, size_t dst_len, const ntr_aov_buffers *aovs);
NTR_API int ntr_group_abort(ntr_group *group);
/* Counters of the last frame summed over the devices; device time of the last frame from the first kernel to the last
 * one of the slowest device (CUDA events on the first device's stream, which waits for the others). */
NTR_API int ntr_group_get_counters(ntr_group *group, ntr_counters *out);
NTR_API int ntr_group_last_kernel_ms(ntr_group *group, float *ms_out);
NTR_API uint64_t ntr_group_launch_count(ntr_group *group);

/* One process per GPU (torchrun): the frame buffer lives in the process of rank 0 and the other ranks store into it
 * through a CUDA IPC mapping -- ntr_frame_alloc + ntr_frame_export on rank 0, ntr_frame_import on the others, then
 * ntr_render_device(scene, fmt, frame, len, stream, rank, world, 0) on every rank (compact = 0: rows at their frame
 * position) and a stream-ordered barrier of the caller's choice (bench.py: a 4-byte NCCL all-reduce). */
#define NTR_IPC_HANDLE_BYTES 64
NTR_API int ntr_frame_alloc(int device, size_t bytes, void **dev_ptr_out);
NTR_API int ntr_frame_free(int device, void *dev_ptr);
NTR_API int ntr_frame_export(void *dev_ptr, unsigned char handle_out[NTR_IPC_HANDLE_BYTES]);
NTR_API int ntr_frame_import(int device, const unsigned char handle[NTR_IPC_HANDLE_BYTES], void **dev_ptr_out);
NTR_API int ntr_frame_release(int device, void *imported_ptr);
/* Fills a frame with one byte value (cudaMemsetAsync; e.g. a background the renderers leave alone outside their rows). */
NTR_API int ntr_frame_fill(int device, void *dev_ptr, int value, size_t bytes, void *stream);
/* device frame -> host buffer (pixel bytes of every row; the pitch padding of dst is left alone), stream-ordered. */
NTR_API int ntr_frame_download(int device, const void *dev_ptr, const ntr_image_format *fmt, void *dst, size_t dst_len, void *stream);

/* ---- control --------------------------------------------------------------------------------- */
/* renderer::state = CANCEL (src/render.cpp:333,412,702-722,911-923): polled per tile on the device. */
NTR_API int ntr_abort(ntr_scene *scene);
/* Counters of the last render call.  `instrumented` renders (ntr_set_instrumented) also fill
 * node_steps / simplex_tests / solid_tests; they are slower and never used for timing. */
NTR_API int ntr_get_counters(ntr_scene *scene, ntr_counters *out);
NTR_API int ntr_set_instrumented(ntr_scene *scene, int on);
/* Device time of the kernels of the last render call in milliseconds (CUDA events on the launching stream). */
NTR_API int ntr_last_kernel_ms(ntr_scene *scene, float *ms_out);
/* Number of kernel launches issued by this library on behalf of `scene` since creation. */
NTR_API uint64_t ntr_launch_count(ntr_scene *scene);

/* ---- scene construction next to the path (SURVEY.md section 8f rows 1-2; host-side, no GPU needed) ---------- */
/* Triangle.from_points / TrianglePrototype for n simplexes at once (src/tracer.hpp:442-462: generalized cross
 * products, src/geometry.hpp:858-893).  points: n x D x D (D vertices each); records: n x ((D+1)*D+1) in the
 * ntr_scene_desc.simplex layout (face_normal[D], d, p1[D], edge_normals[D-1][D]). */
NTR_API int ntr_simplex_from_points(int dim, uint32_t n, const float *points, float *records);
/* k-d tree over n axis-aligned item bounds (lo/hi: n x D), replacing build_kdtree (src/tracer.hpp:1930-2455; kwargs
 * max_depth, split_threshold, traversal_cost, intersection_cost of src/ntracer_body.hpp:3252-3298; <= 0 / < 0 select
 * the defaults 25, 2, 1, 4).  Own algorithm (binned SAH, all axes, straddlers on both sides, empty children null).
 * Outputs are malloc'ed, release them with ntr_free: nodes (leaf w1/w2 index into refs), refs = ITEM INDICES per
 * leaf (0..n-1; the caller maps them to leaf refs), root (NTR_NULL_NODE if n == 0), boundary = 2 x D. */
NTR_API int ntr_build_kdtree(int dim, uint32_t n, const float *lo, const float *hi, int max_depth, int split_threshold,
                             float traversal_cost, float intersection_cost, ntr_node **nodes_out, uint32_t *n_nodes_out,
                             uint32_t **refs_out, uint32_t *n_refs_out, uint32_t *root_out, float *boundary_out);
/* The same tree build with the simplexes behind the items, so that an item is listed only in the cells its geometry
 * can touch -- what the reference's builder achieves with its exact primitive / box overlap tests
 * (src/tracer.hpp:1465-1675, used by split_kdtree :2284-2354) and bounding boxes alone cannot.  Item i owns simplexes
 * item_first[i] .. item_first[i+1]-1 (item_first: n + 1 entries, [0] = 0; an item with none, e.g. a solid, is kept by its
 * bounds); per simplex: bounds s_lo / s_hi (n_simplex x D) and its record (s_records: n_simplex x ((D+1)*D+1), the
 * ntr_scene_desc.simplex layout).  A cell is dropped for a simplex when a separating axis exists among the box axes,
 * the face normal and the D facet directions (the barycentric functions of the ray test, src/tracer.hpp:411-440, are
 * affine: their ranges over the cell come from its extreme corners); conservative by a relative margin.
 * item_first == NULL: ntr_build_kdtree. */
NTR_API int ntr_build_kdtree_culled(int dim, uint32_t n, const float *lo, const float *hi, const uint32_t *item_first,
                                    uint32_t n_simplex, const float *s_lo, const float *s_hi, const float *s_records,
                                    int max_depth, int split_threshold, float traversal_cost, float intersection_cost,
                                    ntr_node **nodes_out, uint32_t *n_nodes_out, uint32_t **refs_out, uint32_t *n_refs_out,
                                    uint32_t *root_out, float *boundary_out);
NTR_API void ntr_free(void *p);
/* Batch grouping ahead of the tree build (group_primitives, src/tracer.hpp:2395-2427: triangles are packed into
 * triangle_batch items of v_real::size lanes).  order_out receives a permutation of the n items (bounds lo/hi: n x D)
 * in which every consecutive run of `group` entries is one batch of spatially close items; the last n % group entries
 * stay single primitives.  Own algorithm: recursive median split of the item centres, O(n log n). */
NTR_API int ntr_group_items(int dim, uint32_t n, const float *lo, const float *hi, int group, uint32_t *order_out);

/* FP32 FMA peak micro-benchmark (TFLOP/s) on the scene's device: the roofline denominator the
 * north star asks for (MEASURED_PEAKS.json has HBM and BF16 only). */
NTR_API int ntr_measure_fp32_peak(int device, float *tflops_out);

#ifdef __cplusplus
}
#endif
#endif /* NTRACER_B200_H */
