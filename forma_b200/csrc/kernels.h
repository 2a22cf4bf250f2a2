// Host-callable launchers of the CUDA kernels (implemented in kernels_*.cu).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "device_types.h"

namespace forma {

// Schedule switches (none of them changes results). Initialised from the environment
// (FORMA_<NAME>) on first use and settable at run time through forma_set_option(), which is
// how the parity tests cover every value (tests/test_gpu_options.py).
struct Options {
    int speculate = 1;       // launch kernels ahead of their count read-backs (0: strictly after)
    int band_copy = 1;       // host frames: paint / copy back in bands of tile rows
    int copy_bands = 4;      //   ... how many (1..16; paris@4K end to end, r2 final build: 4 -> 582.7, 8 -> 567.9, 16 -> 553.8 frames/s; cubics100k 303.6 / 298.6 / 291.1; circles8k 102.3 / 101.1 / 97.7)
    int sort_full_key = 0;   // 1: sort the layer digits even when the inserts are in layer order
    int sort_big_log2 = 19;  // key count from which the 4096-key tiles / reduce-then-scan passes are used
    int sort_scan_log2 = 22; // key-only sorts: key count from which the reduce-then-scan passes replace the single-sweep ones (measured on paris@4K bands: 0.7 M keys 0.044 vs 0.055 ms, 3 M equal, 5.9 M 0.130 vs 0.105 ms)
    int test_gap_cap = 0;    // test hook: cap of the speculative carry-only-entry launch (0 = none)
    int paint_lpt = 1;       // heavy tiles first (longest-processing-time order) in the paint kernel
    int paint_wide = 0;      // 1: the paint kernel built for 6 CTAs / SM (up to 168 registers) instead of 8 (128)
    int band_filter = 1;     // a render cropped to a band of rows only makes the band's geometry resident
    int sync_free = 1;       // painter tables without count read-backs when the previous frame's counts bound this one's (redone the slow way if they do not)
    int test_fast_shrink = 0;  // test hook: halve the bounds of the sync-free tables (forces the redo)
    int host_slices = 1;     // host frames: > 1 = that many tile-row slices rendered as independent upload -> render -> copy-back pipelines on their own streams.
                             //   Off by default: measured on paris@4K 578.9 (off) vs 544-587 frames/s (2-4 slices), 509 (6), 422 (8); cubics100k 298.6 vs 280 / 237;
                             //   the slices' kernel chains do not overlap on the device (latency-bound kernels that fill the SMs), see DESIGN.md section 3
    int slice_bands = 2;     //   ... copy bands inside a slice
    int slice_min_points = 65536;  //   ... only for compositions of at least this many points
    int slice_chain = 1;     //   ... uploads issued slice after slice, each waiting for the one before (0: all at once from the slices' threads)
};
Options& options();

// Arguments of the fused line-setup + pixel-grid-intersection kernels.
struct RasterArgs {
    const float* x;            // segment buffer (segment.rs:530-534)
    const float* y;
    const uint32_t* gid;       // geometry id per point, 0 = None
    uint32_t n_points;
    const int32_t* geom_slot;  // geom id -> layer slot, -1 = not in the composition
    uint32_t n_geoms;
    const LayerRec* layers;    // nullptr when no layer has a transform: then ...
    const uint32_t* layer_bits;// ... order | enabled << 21 per layer slot
    float width, height;       // render target in pixels
    float band_lo, band_hi;    // pixel rows painted by this GPU ([0, height) on one GPU)
};

// ---- kernels_raster.cu ------------------------------------------------------
void launch_flatten_eval(const SplineRec* splines, const PointRec* points, const uint8_t* kinds, const QuadRec* quads,
                         const FlattenJob* jobs, const JobXf* xfs, uint32_t n_jobs, uint32_t n_points,
                         uint32_t dst_base /* first point of the batch in the segment buffer */, float* x, float* y, uint32_t* gid,
                         cudaStream_t stream);
// Rebuilds the device-resident QuadRecs from the uploaded control points (quad_math.h).
void launch_quad_expand(const QuadUp* in, QuadRec* out, uint32_t n, cudaStream_t stream);
void launch_quad_expand_poly(const QuadUpPoly* in, QuadRec* out, uint32_t n, cudaStream_t stream);  // all weights 1
uint32_t raster_num_blocks(uint32_t n_points);
// block_sums: raster_num_blocks(n) entries, turned into exclusive offsets; total[0] = #segments.
// max_tile[0..1] = largest biased tile_x / tile_y any emitted segment can carry.
void launch_line_count(const RasterArgs& args, uint32_t* block_sums, uint32_t* total, uint32_t* max_tile,
                       cudaStream_t stream);
// Segments at positions >= cap are dropped (speculative launches, see Renderer::rasterize).
void launch_raster_emit(const RasterArgs& args, const uint32_t* block_offsets, uint64_t* out, uint32_t cap, cudaStream_t stream);
// Line records of the n = n_points - 1 point pairs (inspection only): orders, then
// f = {x0, y0, dx, dy, a, b, c, d}, then the per-line segment counts.
void launch_line_records(const RasterArgs& args, uint32_t n, uint32_t* orders, float* const f[8], uint32_t* lengths,
                         cudaStream_t stream);
// In-place exclusive scan of n u32 values; total[0] = sum. `state` (scan_state_words(n)
// u64 words) enables the multi-CTA look-back scan for large n; nullptr = one CTA.
size_t scan_state_words(uint32_t n);
// `n_dev` (optional): the element count in device memory, `n` then being its upper bound.
void launch_scan_u32(uint32_t* data, uint32_t n, uint32_t* total, unsigned long long* state, cudaStream_t stream,
                     const uint32_t* n_dev = nullptr);

// ---- kernels_sort.cu --------------------------------------------------------
// LSD radix sort of u64 keys on bits [kSortShift, 64) (+ optional u32 payload).
// Sorted data ends up in keys / vals; *_tmp are same-sized scratch buffers.
// `scratch` needs radix_scratch_bytes(n) bytes. Launch count is returned.
// The 44 ordering bits are three fields; pos/maxw list them from least to most
// significant. Only the low bits of each field that are set in some key (OR of
// all keys | extra_or) take part in the sort passes.
struct KeyLayout {
    uint32_t pos[3];
    uint32_t maxw[3];
};
inline KeyLayout segment_key_layout() { return KeyLayout{{20, 41, 53}, {21, 12, 11}}; }   // ty | tx | layer
inline KeyLayout carry_key_layout() { return KeyLayout{{20, 32, 53}, {12, 21, 11}}; }     // ty | layer | tx

constexpr int kMaxSortPasses = 6;  // ceil(44 / 8)
// One digit = up to three bit runs of the key, concatenated.
struct DigitSpec {
    uint8_t shift[3];
    uint8_t width[3];
    uint8_t lsh[3];
    uint8_t bits;
};
struct SortPlan {
    uint32_t n_passes;
    uint32_t total_bits;
    DigitSpec pass[kMaxSortPasses];
};
// bound[f] = largest value field f (least significant first) takes in any key.
SortPlan make_sort_plan(const KeyLayout& layout, const uint64_t bound[3]);
struct SortResult {
    int launches;
    bool in_tmp;  // the sorted data is in keys_tmp / vals_tmp (odd number of passes)
    int timed_passes = 0;  // passes whose kernels were bracketed by pass_events
};
size_t radix_scratch_bytes(uint32_t n);
SortResult launch_radix_sort(uint64_t* keys, uint64_t* keys_tmp, uint32_t* vals, uint32_t* vals_tmp, uint32_t n,
                             const SortPlan& plan, void* scratch, cudaStream_t stream,
                             cudaEvent_t* pass_events = nullptr /* 3 per pass: before upsweep, before / after downsweep */,
                             const uint32_t* n_dev = nullptr /* the key count in device memory; `n` is then its upper bound
                                                                (single-sweep passes only) */);

// ---- kernels_paint.cu -------------------------------------------------------
struct PaintScene {
    const StyleRec* styles;       // indexed by style slot
    const int32_t* order_to_style;// layer id (order) -> style slot
    uint32_t n_orders;
    const StopRec* stops;
    const GradRec* grads;         // per style slot (valid where the style is a gradient of <= 4 stops)
    const uint16_t* texels;       // RGBA f16 (styling.rs:224-249), 4 per texel
    float clear[4];
    uint32_t channels[4];         // already upgraded Alpha -> One when clear.a == 1
    uint32_t width, height;       // pixels
    uint32_t stride;              // bytes
    uint32_t tiles_x, tiles_y;    // ceil(width / 16), ceil(height / 16)
    uint32_t tx_lo, tx_hi;        // tile columns painted (crop), [lo, hi)
    uint32_t ty_lo, ty_hi;        // tile rows painted (crop ∩ band), [lo, hi)
    // Layer cache (damage reuse, cpu/buffer/mod.rs:114-197); all null/0 without a cache.
    const uint8_t* unchanged;     // per layer order: Layer::is_unchanged(cache_id)
    uint2* cache_tiles;           // per tile: x = has_count<<31 | has_solid<<30 | layer_count(24), y = solid colour
    uint32_t* written_list;       // optional: linear ids of the tiles this frame wrote (unordered)
    uint32_t* written_count;      //           ... and how many
    uint32_t clear_unchanged;     // previous clear colour == this frame's
};

// Output buffer of a frame: format and, for float formats with a layer cache, the per-tile solid
// colour at output precision (4 x f32 bits, or 4 x f16 in .x / .y; PaintScene::cache_tiles[].y is
// unused then). Kept out of PaintScene so that the RGBA8 paint kernel's parameters stay as they were.
struct FrameOut {
    uint32_t format = 0;                // kFormat*
    uint4* cache_solid_wide = nullptr;  // null without a cache and for RGBA8
};

// Output formats of the frame buffer (= FORMA_FORMAT_* in include/forma_b200.h).
constexpr uint32_t kFormatRgba8 = 0, kFormatRgba16f = 1, kFormatRgba32f = 2;
__host__ __device__ constexpr uint32_t format_bytes_per_pixel(uint32_t f) {
    return f == kFormatRgba32f ? 16u : (f == kFormatRgba16f ? 8u : 4u);
}
__host__ __device__ constexpr uint32_t format_element_bytes(uint32_t f) {
    return f == kFormatRgba32f ? 4u : (f == kFormatRgba16f ? 2u : 1u);
}

uint32_t cell_num_blocks(uint32_t n);
// Cells in one pass over the sorted segments (+ a small kernel for the cells that cross a
// CTA tile): cell_start[c] = first segment of cell c (cell_start[#cells] = n), the cell's
// cover (16 x i8 by local_y), its key, the (tile_y, layer, tile_x) key of the carry pass and
// perm[c] = c, for every c < cap - 1; n_cells_out[0] = #cells. All five arrays need `cap`
// entries. `state`: cells_state_words(n) u64 words. May be launched before the host knows the
// count; the caller repeats it if #cells >= cap.
size_t cells_state_words(uint32_t n);
void launch_cells(const PaintScene& S, const uint64_t* segs, uint32_t n, unsigned long long* state, uint32_t* cell_start,
                  uint32_t cap, uint32_t* n_cells_out, uint64_t* cell_key, uint4* cell_cover, uint64_t* key2, uint32_t* perm,
                  cudaStream_t st);
// Plans of the painter's two pair sorts (their key bounds are host-known).
SortPlan carry_sort_plan(const PaintScene& S);
SortPlan gap_sort_plan(const PaintScene& S);
// Cell / carry-only-entry counts that stay on the device (frames whose tables are built without a
// host read-back, Options::sync_free): with `cells` set, the n_cells / n_gaps arguments of the
// launchers below are upper bounds (grid sizes) and the kernels read the counts here; a count
// above its bound makes them no-ops (the host then rebuilds the tables with known counts).
struct DevCounts {
    const uint32_t* cells = nullptr;
    const uint32_t* gaps = nullptr;
    uint32_t cell_bound = 0, gap_bound = 0;
};
void launch_carry_scan(const PaintScene& S, const uint64_t* key2, const uint32_t* perm, const uint4* cell_cover,
                       uint32_t n_cells, uint4* carry_in, uint4* carry_after, uint32_t* gap_count, cudaStream_t st,
                       const DevCounts& dc = DevCounts());
// Carry-only entries in (layer, tile_y, tile_x) order; payload = n_cells + gap id.
void launch_gap_fill(const PaintScene& S, const uint64_t* key2, const uint32_t* perm, const uint64_t* cell_key,
                     const uint4* carry_after, const uint32_t* gap_offset /* scanned gap counts */, uint32_t n_cells,
                     uint64_t* gkey, uint32_t* gid, uint4* gap_carry, const uint32_t* n_gaps_ptr, uint32_t cap,
                     uint32_t grid_gaps /* threads to launch: >= the entry count */, cudaStream_t st,
                     const DevCounts& dc = DevCounts());
// One painter entry = one (tile, layer) pair with segments and / or a carried cover.
struct EntryRec {  // 64 B
    uint32_t layer, seg0, seg1;  // layer order; [seg0, seg1) in the sorted segments (empty for carry-only entries)
    uint32_t meta;               // packed style bits, see pack_style_meta (paint_common.cuh)
    uint4 carry;                 // 16 x i8 cover carried in from the tiles on the left
    float color[4];              // solid fill colour
    int32_t slot;                // style slot
    uint32_t clip_layers;
    uint32_t flags0;             // initial optimizer flags (kFlag*)
    uint32_t pad;
};
// Merges the cells with the sorted carry-only entries: ekey, entry records and
// initial flags of the n_cells + n_gaps entries, ordered by (tile_y, tile_x, layer).
void launch_merge_entries(const PaintScene& S, const uint64_t* cell_key, uint32_t n_cells, const uint64_t* gkey,
                          const uint32_t* gid, uint32_t n_gaps, const uint32_t* cell_start, const uint4* carry_in,
                          const uint4* gap_carry, uint64_t* ekey, EntryRec* recs, uint8_t* eflags, cudaStream_t st,
                          const DevCounts& dc = DevCounts());
// Per-tile entry ranges (zero for tiles without entries) and, when `heavy` is not null, the
// lists of tiles with many entries: kHeavyListClasses arrays of tiles_x * tiles_y ids each,
// their lengths in heavy_count[kHeavyListClasses] (both written here).
constexpr int kHeavyListClasses = 4;
void launch_tile_index(const PaintScene& S, const uint64_t* ekey, uint32_t n_entries, uint2* tile_range, uint32_t* heavy,
                       uint32_t* heavy_count, cudaStream_t st, const DevCounts& dc = DevCounts());
void launch_paint(const PaintScene& S, const uint64_t* segs, const EntryRec* recs, const uint2* tile_range, const uint32_t* heavy,
                  const uint32_t* heavy_count, uint8_t* eflags, uint8_t* framebuffer, uint32_t* tile_counter, cudaStream_t st,
                  const FrameOut& out = FrameOut());
// GradRec of every style slot (see device_types.h).
void launch_grad_setup(const StyleRec* styles, const StopRec* stops, uint32_t n_styles, GradRec* grads, cudaStream_t st);
// Packed fp32 (f32x2) arithmetic of the painter against scalar IEEE operations; mismatches are added to out[0].
void launch_f32x2_selftest(const float* a, const float* b, const float* c, uint32_t n, uint32_t* out, cudaStream_t st);
// out[row] = 32 x entries + pixel segments of tile row `row` (see row_cost_kernel).
void launch_row_costs(const uint2* tile_range, uint32_t tiles_x, uint32_t tiles_y, const uint64_t* segs, uint32_t n,
                      unsigned long long* out, cudaStream_t st, unsigned long long* seg_out = nullptr);
// Packs the tiles in S.written_list into `packed` (256 pixels of `format` per tile, row-major).
void launch_gather_tiles(const PaintScene& S, uint32_t format, const uint8_t* framebuffer, void* packed, cudaStream_t st);

}  // namespace forma
