/*
 * forma_b200 — C ABI of the B200-native replacement for google/forma's
 * rendering hot path (flatten -> pixel-grid intersection -> 64-bit
 * pixel-segment sort -> per-tile paint).
 *
 * The reference has no Renderer trait (SURVEY.md F1); the drop-in boundary is
 * the inherent method forma/src/cpu/renderer.rs:75-82
 *
 *     cpu::Renderer::render(&mut self, composition, buffer, channels,
 *                           clear_color, crop)
 *
 * together with the scene-building API its callers use
 * (forma/src/lib.rs:128-154: Composition, Layer, PathBuilder, Path, Order,
 * Props/Style/Fill/Gradient/BlendMode/FillRule/Func, Buffer/LinearLayout,
 * Channel constants). Every function below names the reference item it
 * replaces. Plain pointers and sizes only; no C++ or torch types.
 *
 * Status codes replace the reference's panics / Results.
 */
#ifndef FORMA_B200_H
#define FORMA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------ */
/* Status                                                                   */
/* ------------------------------------------------------------------------ */
enum {
    FORMA_OK = 0,
    FORMA_ERR_INVALID_ARGUMENT = 1, /* assert!/panic in the reference                     */
    FORMA_ERR_ORDER_LIMIT = 2,      /* OrderError::ExceededLayerLimit, utils/order.rs:56-65 */
    FORMA_ERR_CUDA = 3,             /* a CUDA call failed; see forma_last_error()          */
    FORMA_ERR_NO_DEVICE = 4,        /* no usable sm_100 device: there is NO CPU fallback   */
    FORMA_ERR_CAPACITY = 5          /* an internal device buffer could not be grown        */
};

/* Human-readable description of the last failure on the calling thread. */
const char* forma_last_error(void);

/* consts.rs:25-26,106-108 */
#define FORMA_MAX_WIDTH 65536u
#define FORMA_MAX_HEIGHT 32768u
#define FORMA_LAYER_LIMIT 2097151u
#define FORMA_TILE_WIDTH 16u
#define FORMA_TILE_HEIGHT 16u

/* ------------------------------------------------------------------------ */
/* Data model (forma/src/styling.rs)                                        */
/* ------------------------------------------------------------------------ */
typedef struct forma_color { float r, g, b, a; } forma_color; /* styling.rs:28-33 (linear) */

enum { FORMA_FILL_RULE_NON_ZERO = 0, FORMA_FILL_RULE_EVEN_ODD = 1 };          /* styling.rs:64-67   */
enum { FORMA_GRADIENT_LINEAR = 0, FORMA_GRADIENT_RADIAL = 1 };                /* styling.rs:76-79   */
enum { FORMA_FILL_SOLID = 0, FORMA_FILL_GRADIENT = 1, FORMA_FILL_TEXTURE = 2 }; /* styling.rs:368-372 */
enum { FORMA_FUNC_DRAW = 0, FORMA_FUNC_CLIP = 1 };                            /* styling.rs:417-424 */
enum {                                                                        /* styling.rs:378-395 */
    FORMA_BLEND_OVER = 0, FORMA_BLEND_MULTIPLY, FORMA_BLEND_SCREEN, FORMA_BLEND_OVERLAY,
    FORMA_BLEND_DARKEN, FORMA_BLEND_LIGHTEN, FORMA_BLEND_COLOR_DODGE, FORMA_BLEND_COLOR_BURN,
    FORMA_BLEND_HARD_LIGHT, FORMA_BLEND_SOFT_LIGHT, FORMA_BLEND_DIFFERENCE, FORMA_BLEND_EXCLUSION,
    FORMA_BLEND_HUE, FORMA_BLEND_SATURATION, FORMA_BLEND_COLOR, FORMA_BLEND_LUMINOSITY
};
enum {                                                                        /* cpu/channel.rs:35-43 */
    FORMA_CHANNEL_RED = 0, FORMA_CHANNEL_GREEN, FORMA_CHANNEL_BLUE, FORMA_CHANNEL_ALPHA,
    FORMA_CHANNEL_ZERO, FORMA_CHANNEL_ONE
};

/* One (color, stop) pair of GradientBuilder (styling.rs:84-139). stop == -1
 * means "unpositioned" (GradientBuilder::color): it is spread evenly exactly
 * like GradientBuilder::build does. */
typedef struct forma_gradient_stop { forma_color color; float stop; } forma_gradient_stop;

/* Flat form of Props { fill_rule, func: Draw(Style{is_clipped, fill,
 * blend_mode}) | Clip(n) } (styling.rs:397-442). */
typedef struct forma_props {
    uint32_t fill_rule;
    uint32_t func;        /* FORMA_FUNC_*                                        */
    uint32_t clip_layers; /* n of Func::Clip(n)                                  */
    uint32_t is_clipped;
    uint32_t blend_mode;
    uint32_t fill_type;
    forma_color color;    /* Fill::Solid                                         */
    uint32_t gradient_type;
    float start[2], end[2];
    uint32_t n_stops;
    const forma_gradient_stop* stops;
    float tex_transform[6]; /* Texture.transform: ux, uy, vx, vy, tx, ty         */
    uint32_t tex_width, tex_height;
    const float* tex_linear_rgba; /* Image::from_linear_rgba, styling.rs:320-327 */
} forma_props;

/* cpu::Rect::new(horizontal, vertical) in pixels; approximated to the tile
 * grid exactly like cpu/renderer.rs:43-52. */
typedef struct forma_rect { uint64_t hor_start, hor_end, vert_start, vert_end; } forma_rect;

/* Per-stage device times of the last render (the reference's gpu::Timings,
 * gpu/renderer/mod.rs:25-30) plus the sizes the roofline needs. */
typedef struct forma_timings {
    double line_setup_ms, rasterize_ms, sort_ms, paint_ms;
    uint64_t n_lines, n_segments;
} forma_timings;

/* ------------------------------------------------------------------------ */
/* PathBuilder / Path (forma/src/path.rs:670-925)                           */
/* ------------------------------------------------------------------------ */
typedef struct forma_path_builder forma_path_builder;
typedef struct forma_path forma_path;

forma_path_builder* forma_path_builder_new(void);                 /* PathBuilder::new  :783 */
void forma_path_builder_free(forma_path_builder*);
void forma_path_builder_move_to(forma_path_builder*, float x, float y);            /* :788 */
void forma_path_builder_line_to(forma_path_builder*, float x, float y);            /* :816 */
void forma_path_builder_quad_to(forma_path_builder*, float x1, float y1, float x2, float y2); /* :831 */
void forma_path_builder_cubic_to(forma_path_builder*, float x1, float y1, float x2, float y2,
                                 float x3, float y3);                              /* :850 */
void forma_path_builder_rat_quad_to(forma_path_builder*, float x1, float y1, float x2, float y2,
                                    float weight);                                 /* :873 */
void forma_path_builder_rat_cubic_to(forma_path_builder*, float x1, float y1, float x2, float y2,
                                     float x3, float y3, float w1, float w2);      /* :892 */
forma_path* forma_path_builder_build(forma_path_builder*);                         /* :915 */
forma_path* forma_path_transform(const forma_path*, const float m[9]);   /* Path::transform :726 */
void forma_path_free(forma_path*);

/* Flattened polyline of the path (what Path::push_segments_to appends,
 * path.rs:677-723): n points, start_new_contour[i] != 0 marks a contour end.
 * Pointers stay valid until the next call on the same thread. */
int forma_path_segments(forma_path*, const float** x, const float** y,
                        const uint8_t** start_new_contour, uint64_t* n);
/* Host-side facts of the path's flatten program (no GPU needed): [0] output
 * points, [1] quadratics, [2] spline records, [3] point records (one of [2]/[3]
 * is 0: the smaller encoding is kept), [4] 1 if some quadratic is rational,
 * [5] contour ends before the last point. */
void forma_path_program_stats(forma_path*, uint64_t out[6]);

/* ------------------------------------------------------------------------ */
/* Composition / Layer (forma/src/composition/{mod,layer}.rs)               */
/* ------------------------------------------------------------------------ */
typedef struct forma_composition forma_composition;
/* A Layer handle is owned by its Composition and stays valid until
 * forma_layer_drop() or forma_composition_free(). */
typedef struct forma_layer forma_layer;

forma_composition* forma_composition_new(void);                   /* Composition::new mod.rs:60 */
void forma_composition_free(forma_composition*);
forma_layer* forma_composition_create_layer(forma_composition*);  /* mod.rs:65  (detached)      */
/* Composition::insert(Order::new(order)?, layer) mod.rs:121: returns the
 * displaced layer (now detached) or NULL; *status receives FORMA_ERR_ORDER_LIMIT. */
forma_layer* forma_composition_insert(forma_composition*, uint32_t order, forma_layer*, int* status);
forma_layer* forma_composition_remove(forma_composition*, uint32_t order);          /* mod.rs:141 */
forma_layer* forma_composition_get(forma_composition*, uint32_t order);             /* mod.rs:160 */
forma_layer* forma_composition_get_mut_or_insert_default(forma_composition*, uint32_t order,
                                                         int* status);              /* mod.rs:175 */
uint64_t forma_composition_len(forma_composition*);                                 /* mod.rs:115 */
void forma_layer_drop(forma_composition*, forma_layer*);               /* Drop for Layer, layer.rs:355 */

uint64_t forma_layer_geom_id(forma_layer*);                                        /* layer.rs:160 */
int forma_layer_insert(forma_composition*, forma_layer*, forma_path*);             /* layer.rs:90  */
int forma_layer_clear(forma_composition*, forma_layer*);                           /* layer.rs:131 */
int forma_layer_set_is_enabled(forma_composition*, forma_layer*, int enabled);     /* layer.rs:234 */
int forma_layer_is_enabled(forma_layer*);                                          /* layer.rs:207 */
/* GeomPresTransform::try_from([ux, vx, uy, vy, tx, ty]) + Layer::set_transform
 * (math/transform.rs:196-221, layer.rs:289); INVALID_ARGUMENT if it scales up. */
int forma_layer_set_transform(forma_composition*, forma_layer*, const float t[6]);
int forma_layer_set_props(forma_composition*, forma_layer*, const forma_props*);   /* layer.rs:341 */

/* ------------------------------------------------------------------------ */
/* Renderer (forma/src/cpu/renderer.rs:56-224)                              */
/* ------------------------------------------------------------------------ */
typedef struct forma_renderer forma_renderer;
typedef struct forma_layer_cache forma_layer_cache;

/* Renderer::new (:62). Binds to CUDA device `device_ordinal`. Returns NULL and
 * sets forma_last_error() when no sm_100 device is usable. */
forma_renderer* forma_renderer_new(int device_ordinal);
void forma_renderer_free(forma_renderer*);

/* Renderer::create_buffer_layer_cache (:67); NULL when all 32 ids are in use. */
forma_layer_cache* forma_layer_cache_new(forma_renderer*);
void forma_layer_cache_free(forma_renderer*, forma_layer_cache*);
void forma_layer_cache_clear(forma_layer_cache*);                 /* BufferLayerCache::clear */

/* Renderer::render (:75-224) into a caller-owned HOST buffer laid out like
 * LinearLayout::new(width, width_stride, height) (cpu/buffer/layout/mod.rs:168).
 * Uploads what changed in the composition, runs all stages on the device and
 * copies the framebuffer (or, with a cache, only written tiles) back.
 * `timings` may be NULL: the call then does not read its stage events (a dozen event
 * queries); forma_renderer_stage_times still returns them afterwards. */
int forma_renderer_render(forma_renderer*, forma_composition*, uint8_t* buffer, uint64_t width,
                          uint64_t width_stride, uint64_t height, const uint32_t channels[4],
                          const float clear_color[4], const forma_rect* crop /* nullable */,
                          forma_layer_cache* cache /* nullable */, forma_timings* timings /* nullable */);

/* Same contract, but `device_buffer` is a CUDA device pointer on the
 * renderer's device (e.g. a torch tensor's data_ptr()): no device->host copy.
 * With `reuse_geometry` != 0 and an unchanged composition the points/layer
 * tables already resident in HBM are reused (SURVEY.md §8 N3). */
int forma_renderer_render_device(forma_renderer*, forma_composition*, uint8_t* device_buffer,
                                 uint64_t width, uint64_t width_stride, uint64_t height,
                                 const uint32_t channels[4], const float clear_color[4],
                                 const forma_rect* crop, forma_layer_cache* cache,
                                 forma_timings* timings);

/* Output formats of a frame (the *_format calls below; the calls without the suffix are RGBA8).
 *  - RGBA8: sRGB-encoded bytes, what cpu::Renderer writes (compute_srgb, cpu/painter/mod.rs:466-483).
 *  - RGBA32F: per pixel the four f32 values compute_srgb would receive, before any encode: the
 *    painter's linear accumulator as is (not clamped, not (un)premultiplied; alpha linear as in
 *    RGBA8), 16 bytes. A tile the optimiser folds to one solid colour holds that colour (the value
 *    to_srgb_bytes receives, mod.rs:692).
 *  - RGBA16F: the same values as IEEE binary16, round to nearest even (overflow -> +-inf, NaN stays
 *    NaN), 8 bytes: the format of the reference's gpu::Renderer texture (Rgba16Float).
 * Channel order follows `channels` exactly as for bytes (Zero -> 0.0, One -> 1.0, Alpha -> One when
 * clear_color.a == 1). Layout (width_stride in BYTES), crops, partial edge tiles and layer-cache
 * damage follow the RGBA8 rules. A layer cache compares a solid tile's colour with last frame's at
 * the output precision (the halves / the f32 bit patterns), and a frame of another format than the
 * cache's last one starts the cache over, like a new size does.
 * FORMA_ERR_INVALID_ARGUMENT: unknown format, width * bytes_per_pixel > width_stride, or a stride
 * or buffer address that is not a multiple of the element size (2 bytes RGBA16F, 4 bytes RGBA32F). */
enum { FORMA_FORMAT_RGBA8 = 0, FORMA_FORMAT_RGBA16F = 1, FORMA_FORMAT_RGBA32F = 2 };
int forma_renderer_render_format(forma_renderer*, forma_composition*, void* buffer, uint32_t format, uint64_t width,
                                 uint64_t width_stride, uint64_t height, const uint32_t channels[4],
                                 const float clear_color[4], const forma_rect* crop, forma_layer_cache* cache,
                                 forma_timings* timings);
/* The frame stays in HBM: with RGBA16F it is what gpu::Renderer::render_to_texture leaves in its
 * texture, ready for a consumer on the same device (e.g. a torch tensor's data_ptr()). */
int forma_renderer_render_device_format(forma_renderer*, forma_composition*, void* device_buffer, uint32_t format,
                                        uint64_t width, uint64_t width_stride, uint64_t height,
                                        const uint32_t channels[4], const float clear_color[4],
                                        const forma_rect* crop, forma_layer_cache* cache, forma_timings* timings);

/* Launch on `cuda_stream` (a cudaStream_t, e.g. torch.cuda.current_stream().cuda_stream)
 * instead of the default stream. */
void forma_renderer_set_stream(forma_renderer*, void* cuda_stream);

/* Several GPUs behind one renderer, single process (Renderer::new for a multi-GPU box):
 * `render` has the contract of forma_renderer_render, `render_device` that of
 * forma_renderer_render_device with the frame in the FIRST listed device's memory (the other
 * devices store their rows into it over NVLink; needs peer access). The frame is split into
 * bands of tile rows, one per device, rebalanced every frame on the previous frame's row
 * costs; each device keeps only its band's geometry resident. Layer caches are not
 * supported here (cache = NULL semantics). Every listed device must be an sm_100 GPU. */
typedef struct forma_renderer_multi forma_renderer_multi;
forma_renderer_multi* forma_renderer_multi_new(const int* device_ordinals, int n);
void forma_renderer_multi_free(forma_renderer_multi*);
int forma_renderer_multi_device_count(const forma_renderer_multi*);
int forma_renderer_multi_render(forma_renderer_multi*, forma_composition*, uint8_t* buffer, uint64_t width,
                                uint64_t width_stride, uint64_t height, const uint32_t channels[4],
                                const float clear_color[4], const forma_rect* crop, forma_timings* timings);
int forma_renderer_multi_render_device(forma_renderer_multi*, forma_composition*, uint8_t* buffer_on_first_device,
                                       uint64_t width, uint64_t width_stride, uint64_t height,
                                       const uint32_t channels[4], const float clear_color[4],
                                       const forma_rect* crop, forma_timings* timings);
/* The same in any FORMA_FORMAT_* (see forma_renderer_render_format): every device's band lands in
 * the host buffer / the first device's frame at the format's width. */
int forma_renderer_multi_render_format(forma_renderer_multi*, forma_composition*, void* buffer, uint32_t format,
                                       uint64_t width, uint64_t width_stride, uint64_t height,
                                       const uint32_t channels[4], const float clear_color[4],
                                       const forma_rect* crop, forma_timings* timings);
int forma_renderer_multi_render_device_format(forma_renderer_multi*, forma_composition*, void* buffer_on_first_device,
                                              uint32_t format, uint64_t width, uint64_t width_stride, uint64_t height,
                                              const uint32_t channels[4], const float clear_color[4],
                                              const forma_rect* crop, forma_timings* timings);
/* bounds[n + 1]: tile-row boundaries of the bands the next frame will use; band_ms[n]:
 * device-timeline ms of every band in the last frame. Returns n. */
int forma_renderer_multi_bands(const forma_renderer_multi*, uint32_t* bounds, double* band_ms);

/* Multi-GPU frame assembly without a copy (one process per GPU, tile-row bands,
 * SURVEY.md §8e): the process that owns the frame allocates it with
 * forma_shared_frame_create and passes the 64-byte handle to the others (any
 * channel, e.g. torch.distributed); they map it with forma_shared_frame_open
 * (CUDA IPC, peer access over NVLink) and hand the mapped pointer to
 * forma_renderer_render_device with their band as `crop`: the paint kernel's
 * stores then land directly in the owner's HBM. The caller synchronises the
 * ranks (a barrier / 1-element all-reduce on the render streams) before the
 * owner reads the frame. */
typedef struct forma_ipc_handle { unsigned char bytes[64]; } forma_ipc_handle;
int forma_shared_frame_create(int device, uint64_t bytes, void** device_ptr, forma_ipc_handle* handle);
int forma_shared_frame_open(int device, const forma_ipc_handle* handle, void** device_ptr);
int forma_shared_frame_close(int device, void* mapped_ptr); /* a pointer from _open   */
int forma_shared_frame_free(int device, void* device_ptr);  /* a pointer from _create */

/* --- extensions (no reference counterpart) --------------------------------- */
/* Bulk form of move_to/line_to/quad_to/cubic_to: cmds[i] in {0 Move, 1 Line,
 * 2 Quad, 3 Cubic}, xy = the points they consume (1, 1, 2, 3 points each). */
void forma_path_builder_extend(forma_path_builder*, const uint8_t* cmds, uint64_t n_cmds, const float* xy);
/* Drops the composition's device residency: the next render re-uploads every
 * flatten program and table from pinned host memory (cold end-to-end path). */
void forma_composition_evict(forma_composition*);
uint64_t forma_composition_point_count(forma_composition*);
/* Device-timeline milliseconds of the last render: [0] uploads, [1] line-setup
 * count pass, [2] pixel-grid intersection, [3] sort, [4] painter tables,
 * [5] paint kernel, [6] device->host copy, [7] whole call. */
void forma_renderer_stage_times(const forma_renderer*, double out_ms[8]);
/* CUDA-event time of single kernels inside the last render, summed over their
 * launches: [0] radix downsweep (main sort, one launch per pass), [1] radix
 * upsweep + tile scan (one pair per pass), [2] paint kernel, [3] unused. */
void forma_renderer_kernel_times(const forma_renderer*, double out_ms[4], uint32_t out_launches[4]);
/* [0] kernel launches, [1] host->device bytes, [2] device->host bytes (all
 * since creation), [3] pixel segments, [4] cells, [5] entries of the last render,
 * [6] tiles the last layer-cache render copied back to a host buffer, [7] how the last
 * render built its painter tables: 0 = with the cell / entry counts read back on the way,
 * 1 = without a read-back (kernels sized by the previous frame's counts, option sync_free),
 * 2 = attempted without, counts exceeded the bounds, tables and paint repeated as 0. */
void forma_renderer_counters(const forma_renderer*, uint64_t out[8]);
/* Host frames (forma_renderer_render without a layer cache) of compositions whose layers carry no
 * transform are rendered as a pipeline of tile-row slices on the renderer's device (option
 * host_slices): slice k + 1 uploads its band's geometry while slice k computes and slice k - 1
 * copies its rows back. Returns the number of slices of the last host frame (0 = one piece);
 * out_ms (may be null, room for 16) receives each slice's device-timeline ms (from the start of the
 * frame: a slice's upload waits for those of the slices before it), out_stage_ms (may be null,
 * room for 16 x 8) each slice's stage times as in forma_renderer_stage_times. After a sliced
 * frame the counters above are sums over the slices (pixel segments and entries: every slice
 * counts its own rows, so they are the frame's; cells: an upper bound, a slice also sees the
 * segments boundary-crossing lines leave in its neighbours' rows) and the stage times those of
 * the slowest slice. */
int forma_renderer_host_slices(const forma_renderer*, double* out_ms, double* out_stage_ms);

/* Cost of every tile row of the last render (32 x its (tile, layer) entries + its pixel
 * segments; rows outside the rendered crop cost 0): what a caller balances the tile-row
 * bands of the next multi-GPU frame on (SURVEY.md 8e). Returns the number of tile rows;
 * call with cap = 0 to size `out`. */
uint64_t forma_renderer_row_costs(forma_renderer*, uint64_t cap, uint64_t* out);

/* Schedule switches of the library (process-wide; none changes results): "speculate",
 * "band_copy", "copy_bands", "sort_full_key", "sort_big_log2", "sort_scan_log2", "paint_lpt",
 * "paint_wide", "band_filter", "sync_free", "host_slices", "slice_bands", "slice_min_points", "slice_chain",
 * "test_gap_cap", "test_fast_shrink".
 * Defaults come from the environment (FORMA_SPECULATE, ...); see DESIGN.md section 6. */
int forma_set_option(const char* name, int value);
int forma_get_option(const char* name, int* value);

/* Device self-test of the painter's packed-fp32 (f32x2) arithmetic against the scalar IEEE
 * operations it stands for (2^20 operand triples incl. zeros, denormals, infinities, NaN);
 * *mismatches must come back 0. */
int forma_debug_selftest(int device, uint64_t* mismatches);

/* Number of CUDA kernels the renderer launched since it was created. */
uint64_t forma_renderer_launch_count(const forma_renderer*);

/* --- stage-level access (parity tests; the reference's own tests reach the
 *     same data through Rasterizer::segments(), cpu/rasterizer.rs:88) -------- */

/* The line records of the last render (SegmentBufferView of segment.rs:530-545: one
 * record per point pair, `lengths` as inclusive prefix sums) in host arrays of capacity
 * `cap`; returns the count (call with cap = 0 to size the arrays). render() never
 * materialises them; they are recomputed here from the last render's composition, which
 * must still be alive. */
uint64_t forma_renderer_lines(forma_renderer*, uint64_t cap, uint32_t* orders, float* x0, float* y0,
                              float* dx, float* dy, float* a, float* b, float* c, float* d,
                              uint32_t* lengths);
/* Copy the SORTED pixel segments of the last render; returns the count. */
uint64_t forma_renderer_segments(forma_renderer*, uint64_t cap, uint64_t* segments);
/* Line setup + pixel-grid intersection only; copies the UNSORTED segments (in
 * the reference's emission order) to `segments`; returns the count. */
uint64_t forma_renderer_rasterize_only(forma_renderer*, forma_composition*, uint64_t width,
                                       uint64_t height, uint64_t cap, uint64_t* segments);
/* Stage 3 alone: sort `n` host keys on bits [20, 64) on the device
 * (replaces crumsort at cpu/rasterizer.rs:162-164). */
int forma_renderer_sort_u64(forma_renderer*, uint64_t* keys, uint64_t n);

#ifdef __cplusplus
}
#endif
#endif /* FORMA_B200_H */
