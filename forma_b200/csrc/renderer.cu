// forma_b200 — Composition bookkeeping, Renderer::render orchestration and
// the C ABI of include/forma_b200.h.
//
// Renderer::render follows forma/src/cpu/renderer.rs:75-224 stage by stage;
// every stage is a CUDA kernel sequence on one stream, and there is no CPU
// fallback: without a usable sm_100 device forma_renderer_new() fails.
#include <algorithm>
#include <cctype>
#include <condition_variable>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/forma_b200.h"
#include "cuda_common.cuh"
#include "host_scene.hpp"
#include "kernels.h"

namespace forma {

// ---------------------------------------------------------------------------
// Errors
// ---------------------------------------------------------------------------
static thread_local std::string g_error;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
}

// ---------------------------------------------------------------------------
// Options
// ---------------------------------------------------------------------------
struct OptionName {
    const char* name;
    int Options::*field;
    int lo, hi;
};
static const OptionName kOptionNames[] = {
    {"speculate", &Options::speculate, 0, 1},         {"band_copy", &Options::band_copy, 0, 1},
    {"copy_bands", &Options::copy_bands, 1, 16},      {"sort_full_key", &Options::sort_full_key, 0, 1},
    {"sort_big_log2", &Options::sort_big_log2, 10, 30}, {"test_gap_cap", &Options::test_gap_cap, 0, 1 << 30},
    {"paint_lpt", &Options::paint_lpt, 0, 1},         {"band_filter", &Options::band_filter, 0, 1},
    {"paint_wide", &Options::paint_wide, 0, 1},       {"sort_scan_log2", &Options::sort_scan_log2, 10, 31},
    {"sync_free", &Options::sync_free, 0, 1},         {"test_fast_shrink", &Options::test_fast_shrink, 0, 1},
    {"host_slices", &Options::host_slices, 1, 16},    {"slice_bands", &Options::slice_bands, 1, 16},
    {"slice_min_points", &Options::slice_min_points, 0, 1 << 30}, {"slice_chain", &Options::slice_chain, 0, 1},
};
Options& options() {
    static Options o = [] {
        Options v;
        for (const OptionName& n : kOptionNames) {
            std::string env = "FORMA_";
            for (const char* c = n.name; *c; ++c) env += (char)toupper((unsigned char)*c);
            if (const char* e = getenv(env.c_str())) {
                long x = strtol(e, nullptr, 10);
                if (x >= n.lo && x <= n.hi) v.*(n.field) = (int)x;
            }
        }
        return v;
    }();
    return o;
}

// ---------------------------------------------------------------------------
// Props
// ---------------------------------------------------------------------------
static bool same4(const float* a, const float* b, int n) {
    for (int i = 0; i < n; ++i)
        if (!(a[i] == b[i])) return false;
    return true;
}

// Props: PartialEq (styling.rs derives + Gradient/Image impls).
bool HostProps::equals(const HostProps& o) const {
    const StyleRec &a = rec, &b = o.rec;
    if (a.fill_rule != b.fill_rule || a.func != b.func) return false;
    if (a.func == 1u) return a.clip_layers == b.clip_layers;
    if (a.is_clipped != b.is_clipped || a.blend_mode != b.blend_mode || a.fill_type != b.fill_type) return false;
    if (a.fill_type == 0u) return same4(a.color, b.color, 4);
    if (a.fill_type == 1u) {
        if (a.gradient_type != b.gradient_type || !same4(a.start, b.start, 2) || !same4(a.end, b.end, 2) ||
            stops.size() != o.stops.size())
            return false;
        for (size_t i = 0; i < stops.size(); ++i)
            if (!same4(stops[i].color, o.stops[i].color, 4) || !(stops[i].stop == o.stops[i].stop)) return false;
        return true;
    }
    return texels == o.texels && a.tex_max_x == b.tex_max_x && a.tex_max_y == b.tex_max_y &&
           same4(a.tex_xf, b.tex_xf, 6);
}

// ---------------------------------------------------------------------------
// Composition (composition/mod.rs, composition/layer.rs)
// ---------------------------------------------------------------------------
Layer* Composition::create_layer() {  // mod.rs:65-83
    std::unique_ptr<Layer> owned(new Layer());
    Layer* l = owned.get();
    pool.emplace(l, std::move(owned));
    l->geom_id = next_geom_id++;
    l->dense_id = next_dense_id++;
    return l;
}

void Composition::set_order(Layer* l, int64_t order) {  // layer.rs:148-158
    if (order >= 0 && l->order != order) {
        l->order = order;
        l->unchanged_bits = 0;
    }
    geom_to_order[l->dense_id] = order;
    tables_dirty = true;
}

Layer* Composition::insert(uint32_t order, Layer* layer) {  // mod.rs:121-138
    // The reference takes the Layer by value: a layer cannot sit at two orders. Through
    // the C ABI the same handle can be inserted again, which moves it.
    if (layer->order >= 0 && (uint32_t)layer->order != order) {
        auto at = layers.find((uint32_t)layer->order);
        if (at != layers.end() && at->second == layer) layers.erase(at);
    }
    set_order(layer, order);
    Layer* old = nullptr;
    auto it = layers.find(order);
    if (it != layers.end()) {
        old = it->second;
        it->second = layer;
    } else {
        layers.emplace(order, layer);
    }
    if (old == layer) return nullptr;
    if (old) set_order(old, -1);
    return old;
}

Layer* Composition::remove(uint32_t order) {  // mod.rs:141-149
    auto it = layers.find(order);
    if (it == layers.end()) return nullptr;
    Layer* l = it->second;
    layers.erase(it);
    set_order(l, -1);
    return l;
}

Layer* Composition::get(uint32_t order) {
    auto it = layers.find(order);
    return it == layers.end() ? nullptr : it->second;
}

Layer* Composition::get_or_insert_default(uint32_t order) {  // mod.rs:175-182
    Layer* l = get(order);
    if (!l) {
        l = create_layer();
        insert(order, l);
    }
    return l;
}

void Composition::drop(Layer* l) {  // Drop for Layer, layer.rs:355-363
    if (l->order >= 0) {  // attached layers are found by their order; a detached one keeps a stale order
        auto it = layers.find((uint32_t)l->order);
        if (it != layers.end() && it->second == l) layers.erase(it);
    }
    geom_to_order.erase(l->dense_id);
    garbage_points += l->points;
    pool.erase(l);
    tables_dirty = true;
}

// Layer::insert (layer.rs:90-111) + SegmentBuffer::push_path (segment.rs:181-198).
void Composition::layer_insert(Layer* layer, const Path& path) {
    const FlattenProgram& prog = path.data->program();
    uint32_t count = prog.n_points;
    if (count) {
        if ((uint64_t)n_points + count >= (1ull << 32)) compact_geom();  // dead geometry counts until compacted
        if ((uint64_t)n_points + count >= (1ull << 32))
            throw std::length_error("segment buffer would exceed 2^32 points");
        PendingInsert job;
        job.data = path.data;
        job.has_xf = path.has_xf;
        std::memcpy(job.xf, path.xf, sizeof(job.xf));
        job.geom_id = layer->dense_id;
        job.dst = n_points;
        job.count = count;
        // Rows the insert can reach (for the band filter of multi-GPU frames): the program's
        // bounds through the path's transform, widened by half a pixel plus a relative term
        // that covers the rounding of the evaluation; infinite when the hull argument fails.
        job.y_min = -INFINITY;
        job.y_max = INFINITY;
        if (prog.bounded) {
            float lo = prog.min_y, hi = prog.max_y;
            if (path.has_xf) {  // ty = fma(uy, x, fma(vy, y, t.y)) over the four corners
                lo = INFINITY;
                hi = -INFINITY;
                for (int cx = 0; cx < 2; ++cx)
                    for (int cy = 0; cy < 2; ++cy) {
                        const float px = cx ? prog.max_x : prog.min_x, py = cy ? prog.max_y : prog.min_y;
                        const float ty = fmaf(path.xf[1], px, fmaf(path.xf[3], py, path.xf[5]));
                        lo = std::fmin(lo, ty);
                        hi = std::fmax(hi, ty);
                    }
            }
            if (lo == lo && hi == hi && std::isfinite(lo) && std::isfinite(hi)) {
                const float margin = 0.5f + 1e-4f * std::fmax(std::fabs(lo), std::fabs(hi));
                job.y_min = lo - margin;
                job.y_max = hi + margin;
            }
        }
        jobs.push_back(std::move(job));
        // ids that are Some: every point that does not end a contour, except the
        // last point of the insert (its id is the trailing None).
        uint64_t some = (uint64_t)(count - 1u) - prog.n_contour_ends;
        some_ids += some;
        layer->lines_count += some;
        layer->points += count;
        n_points += count;
    }
    geom_to_order[layer->dense_id] = layer->order;
    layer->unchanged_bits = 0;
    tables_dirty = true;
}

void Composition::compact_geom() {
    const bool dead_points = garbage_points >= 65536u && garbage_points * 2u >= n_points;
    const bool dead_ids = (uint64_t)next_dense_id > 2u * (uint64_t)pool.size() + 65536u;
    if (!dead_points && !dead_ids) return;
    // Dense ids are handed out again from 1, in the order the live layers got theirs, so
    // that the device's id -> layer table stays proportional to the live layers however
    // often layers are cleared (every Layer::clear takes a new id, layer.rs:131-146).
    std::vector<Layer*> alive;
    alive.reserve(pool.size());
    for (auto& kv : pool) alive.push_back(kv.first);
    std::sort(alive.begin(), alive.end(), [](const Layer* a, const Layer* b) { return a->dense_id < b->dense_id; });
    std::unordered_map<uint32_t, uint32_t> renumbered;
    std::unordered_map<uint32_t, int64_t> orders;
    renumbered.reserve(alive.size());
    orders.reserve(alive.size());
    uint32_t next = 1;
    for (Layer* l : alive) {
        auto it = geom_to_order.find(l->dense_id);
        if (it != geom_to_order.end()) orders.emplace(next, it->second);
        renumbered.emplace(l->dense_id, next);
        l->dense_id = next++;
    }
    std::vector<PendingInsert> live;
    live.reserve(jobs.size());
    uint64_t pts = 0;
    for (PendingInsert& j : jobs) {
        auto it = renumbered.find(j.geom_id);  // inserts of cleared / dropped geometry have no live id
        if (it == renumbered.end() || !orders.count(it->second)) continue;
        j.geom_id = it->second;
        j.dst = (uint32_t)pts;
        pts += j.count;
        live.push_back(std::move(j));
    }
    jobs.swap(live);
    geom_to_order.swap(orders);
    next_dense_id = next;
    n_points = (uint32_t)pts;
    garbage_points = 0;
    ++geom_epoch;  // everything is evaluated again into the re-packed buffers (see Renderer::flush_geometry)
    tables_dirty = true;
}

void Composition::layer_clear(Layer* layer) {  // layer.rs:131-146
    garbage_points += layer->points;
    layer->points = 0;
    geom_to_order.erase(layer->dense_id);
    layer->geom_id = next_geom_id++;
    layer->dense_id = next_dense_id++;
    geom_to_order[layer->dense_id] = layer->order;
    layer->lines_count = 0;
    layer->unchanged_bits = 0;
    tables_dirty = true;
}

// ---------------------------------------------------------------------------
// Renderer
// ---------------------------------------------------------------------------
// BufferLayerCache (cpu/buffer/mod.rs:114-197). The per-tile records live on the
// device (the painter reads and updates them); the host only keeps the size, output
// format and clear colour of the last frame.
struct LayerCache {
    uint8_t id = 0;
    DeviceBuffer<uint2> tiles;       // CachedTile per tile, see PaintScene::cache_tiles
    DeviceBuffer<uint4> solid_wide;  // float formats: per-tile solid colour at output precision
    bool has_size = false;
    uint64_t width = 0, height = 0;
    uint32_t format = kFormatRgba8;
    bool has_clear = false;
    float clear_color[4] = {0, 0, 0, 0};
    bool needs_reset = true;  // the tile records must be zeroed before their next use
    void clear() {            // BufferLayerCache::clear, mod.rs:189-196
        has_clear = false;
        needs_reset = true;
    }
};

struct Timer {
    cudaEvent_t ev[8];
    cudaEvent_t sort_ev[3 * kMaxSortPasses];  // main sort, per pass: before upsweep, before / after downsweep
    bool ok = false;
};

class Renderer {
   public:
    int device = 0;
    int res_key = 0;  // key of this renderer's residency record in a Composition: the device ordinal, or
                      // device + 4096 * (k + 1) for the k-th slice renderer of a host-frame pipeline
    int copy_bands_override = 0;  // slice renderers: copy bands inside the slice (0 = option copy_bands)
    cudaStream_t stream = 0;
    bool owns_stream = false;
    uint64_t launches = 0;
    uint32_t caches_in_use = 0;
    Timer timer;

    // Per-frame device scratch (high-water-mark allocations).
    DeviceBuffer<uint32_t> block_sums, totals;
    DeviceBuffer<unsigned long long> scan_state;
    SortPlan segment_plan{};  // digits of the main sort, from the bounds seen by the line-setup pass

    template <class T>
    static void swap_buffers(DeviceBuffer<T>& a, DeviceBuffer<T>& b) {
        std::swap(a.ptr, b.ptr);
        std::swap(a.capacity, b.capacity);
    }
    DeviceBuffer<uint64_t> segs, segs_tmp;
    DeviceBuffer<uint8_t> sort_scratch;
    DeviceBuffer<uint32_t> cell_start, perm, perm_tmp, gap_count, eid, eid_tmp, gid_tmp, heavy_tiles;
    DeviceBuffer<uint2> tile_range;
    DeviceBuffer<uint64_t> cell_key, key2, key2_tmp, ekey, ekey_tmp, gkey_tmp;
    DeviceBuffer<uint4> cell_cover, carry_in, carry_after, gap_carry;
    DeviceBuffer<uint8_t> eflags, framebuffer;
    DeviceBuffer<EntryRec> recs;
    // Band-wise copy-back of host frames (see render()).
    static constexpr uint32_t kMaxCopyBands = 16;
    uint32_t copy_bands() const {
        return (uint32_t)std::min(std::max(copy_bands_override ? copy_bands_override : options().copy_bands, 1), (int)kMaxCopyBands);
    }
    cudaStream_t aux_stream = nullptr;  // side stream of the geometry upload (see flush_geometry)
    cudaEvent_t aux_ev[2];
    cudaStream_t band_stream[kMaxCopyBands];
    uint32_t band_streams_made = 0;  // created as needed: streams beyond the device's hardware queues alias onto them
    bool band_streams_ok = false;    // the band events exist
    cudaEvent_t band_ev[kMaxCopyBands + 1];
    cudaEvent_t count_ev = nullptr;  // completion of a count read-back (waited on instead of the whole stream)
    cudaError_t ensure_count_event() {
        return count_ev ? cudaSuccess : cudaEventCreateWithFlags(&count_ev, cudaEventDisableTiming);
    }
    static bool speculation_enabled() { return options().speculate != 0; }
    static size_t test_gap_cap_override() { return (size_t)std::max(options().test_gap_cap, 0); }
    static bool band_copies_enabled() { return options().band_copy != 0; }
    // Layer-cache frames: per-slot `is_unchanged` flags, the list of written
    // tiles and their packed pixels (only these travel back to a host buffer).
    DeviceBuffer<uint8_t> d_unchanged;
    PinnedBuffer<uint8_t> h_unchanged;
    DeviceBuffer<uint32_t> written_list, packed_tiles;
    PinnedBuffer<uint32_t> h_written_list, h_packed_tiles;
    uint32_t last_written_tiles = 0;
    // Upload staging.
    DeviceBuffer<QuadUp> up_quads_raw;  // as uploaded; expanded into up_quads on the device
    DeviceBuffer<SplineRec> up_splines;
    DeviceBuffer<PointRec> up_points;
    DeviceBuffer<uint8_t> up_kinds;
    DeviceBuffer<QuadRec> up_quads;
    DeviceBuffer<FlattenJob> up_jobs;
    DeviceBuffer<JobXf> up_xfs;

    uint32_t last_segments = 0, last_cells = 0, last_entries = 0, last_gaps = 0;
    bool last_tables_sync_free = false, last_tables_redone = false;  // how the last frame's painter tables were built
    uint32_t last_tiles_x = 0, last_tiles_y = 0;  // tile grid of the last render (forma_renderer_row_costs)
    RasterArgs last_raster{};        // line-setup arguments of the last render (device pointers owned by its composition)
    bool last_raster_valid = false;
    uint64_t h2d_bytes = 0, d2h_bytes = 0;  // bytes copied over PCIe since creation
    double stage_ms[8] = {0};               // see forma_renderer_stage_times (valid after resolve_times)
    double kernel_ms[4] = {0};              // see forma_renderer_kernel_times
    uint32_t kernel_launches[4] = {0};
    bool times_pending = false;             // the last render's events have not been turned into stage_ms / kernel_ms yet
    int pending_sort_passes = 0;
    uint32_t pending_paint_launches = 0;
    void resolve_times() {
        if (!times_pending || !timer.ok) return;
        times_pending = false;
        cudaSetDevice(device);
        auto el = [&](int a, int b) {
            float ms = 0;
            cudaEventElapsedTime(&ms, timer.ev[a], timer.ev[b]);
            return (double)ms;
        };
        stage_ms[0] = el(0, 7);  // uploads (geometry programs + flatten eval + tables)
        stage_ms[1] = el(7, 1);  // line setup: count pass + scan (+ count read-back)
        stage_ms[2] = el(1, 2);  // pixel-grid intersection (emit)
        stage_ms[3] = el(2, 3);  // sort (upsweep / tile scan / downsweep per digit), no host sync inside
        stage_ms[4] = el(3, 4);  // painter tables: cells, carries, entries (2 pair sorts)
        stage_ms[5] = el(4, 5);  // paint kernel alone (host frames: its band launches)
        stage_ms[6] = el(5, 6);  // device -> host copy of the framebuffer
        stage_ms[7] = el(0, 6);  // whole call on the device timeline
        kernel_ms[0] = kernel_ms[1] = 0;
        for (int p = 0; p < pending_sort_passes; ++p) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, timer.sort_ev[3 * p], timer.sort_ev[3 * p + 1]);
            cudaEventElapsedTime(&b, timer.sort_ev[3 * p + 1], timer.sort_ev[3 * p + 2]);
            kernel_ms[1] += a;  // upsweep + tile scan
            kernel_ms[0] += b;  // downsweep
        }
        kernel_launches[0] = kernel_launches[1] = (uint32_t)pending_sort_passes;
        kernel_ms[2] = stage_ms[5];
        kernel_launches[2] = pending_paint_launches;
    }
    uint32_t* pinned_totals = nullptr;  // 4 x u32 pinned host words for count read-backs
    // Renderers of a multi-device / sliced frame: the per-row costs of the frame (see
    // row_cost_kernel) travel back behind the frame itself, without a synchronisation of their own.
    bool track_row_costs = false;
    DeviceBuffer<unsigned long long> d_row_costs;
    PinnedBuffer<unsigned long long> h_row_costs;
    uint32_t row_costs_rows = 0;  // rows of h_row_costs that belong to the last render (0 = none)
    uint32_t last_slices = 0;     // slices of the last host frame (0 = rendered as one piece)
    // Slice renderers of a host-frame pipeline: the uploads of the slices are issued by one thread,
    // slice after slice, and chained (a slice's copies wait for the previous slice's), so that slice k
    // has its geometry - and starts computing - while slices k + 1 ... are still crossing PCIe.
    cudaEvent_t upload_done_ev = nullptr;  // recorded behind this renderer's last host -> device copy
    cudaEvent_t upload_after = nullptr;    // this renderer's copies wait for it (the previous slice's upload_done_ev)
    bool prefetched = false;               // prefetch() ran for the coming render: timer.ev[0] is already recorded
    int prefetch(Composition& comp, uint64_t width, uint64_t height, const forma_rect* crop);
    int ensure_timer() {
        if (!timer.ok) {
            for (auto& e : timer.ev) FORMA_CUDA_TRY(cudaEventCreate(&e));
            for (auto& e : timer.sort_ev) FORMA_CUDA_TRY(cudaEventCreate(&e));
            timer.ok = true;
        }
        return FORMA_STATUS_OK;
    }

    ~Renderer() {
        if (pinned_totals) cudaFreeHost(pinned_totals);
        if (count_ev) cudaEventDestroy(count_ev);
        if (upload_done_ev) cudaEventDestroy(upload_done_ev);
        if (band_streams_ok)
            for (auto& e : band_ev) cudaEventDestroy(e);
        for (uint32_t k = 0; k < band_streams_made; ++k) cudaStreamDestroy(band_stream[k]);
        if (timer.ok) {
            for (auto& e : timer.ev) cudaEventDestroy(e);
            for (auto& e : timer.sort_ev) cudaEventDestroy(e);
        }
        if (aux_stream) {
            cudaEventDestroy(aux_ev[0]);
            cudaEventDestroy(aux_ev[1]);
            cudaStreamDestroy(aux_stream);
        }
        if (owns_stream && stream) cudaStreamDestroy(stream);
    }

    int flush_geometry(Composition& comp, float band_lo = 0.0f, float band_hi = 0.0f, bool band_is_partial = false);
    int upload_tables(Composition& comp, int64_t cache_id);
    static int rebuild_tables(Composition& comp, int64_t cache_id);
    int upload_tables_device(Composition& comp, CompDevice& cd);
    int read_total(uint32_t slot, uint32_t* out);
    int rasterize(Composition& comp, uint32_t width, uint32_t height, float band_lo, float band_hi, uint32_t* n_out);
    int render(Composition& comp, uint8_t* buffer, bool buffer_on_device, uint64_t width, uint64_t stride,
               uint64_t height, const uint32_t channels[4], const float clear[4], const forma_rect* crop,
               LayerCache* cache, forma_timings* timings, uint32_t format = kFormatRgba8);
};

int Renderer::read_total(uint32_t slot, uint32_t* out) {
    FORMA_CUDA_TRY(cudaMemcpyAsync(pinned_totals + slot, totals.ptr + slot, sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                   stream));
    FORMA_CUDA_TRY(cudaStreamSynchronize(stream));
    *out = pinned_totals[slot];
    return FORMA_STATUS_OK;
}

static QuadUp quad_upload(const QuadRec& q) {
    QuadUp u;
    for (int k = 0; k < 3; ++k) {
        u.px[k] = q.px[k];
        u.py[k] = q.py[k];
        u.pw[k] = q.pw[k];
    }
    u.prev_curv = q.prev_curv;
    u.total = q.total;
    u.step = q.step;
    return u;
}

// Evaluates the Layer::insert jobs that are not resident on this device yet into its
// segment buffer: one batched upload from pinned staging + one kernel. With a band
// ([band_lo, band_hi) in pixel rows, narrower than the frame) and no layer transform in
// the composition, inserts that cannot reach the band are left out: a GPU that paints a
// band of tile rows then uploads, evaluates and scans only the geometry of its band.
int Renderer::flush_geometry(Composition& comp, float band_lo, float band_hi, bool band_is_partial) {
    comp.compact_geom();
    CompDevice& cd = comp.on(res_key);
    if (cd.geom_epoch != comp.geom_epoch) {  // compacted since: the resident points are stale
        cd.reset_residency();
        cd.geom_epoch = comp.geom_epoch;
    }
    // The filter only holds while no layer moves its geometry (a layer transform would have to be
    // applied to the bounds, and changes from frame to frame): fall back to everything otherwise.
    // (comp.layers_have_xf is maintained by rebuild_tables, which every caller runs first.)
    const bool want_filter = band_is_partial && !comp.layers_have_xf && options().band_filter != 0;
    if (cd.jobs_resident > 0) {
        // What is resident must cover what this render needs.
        const bool covers = !cd.filtered || (want_filter && band_lo >= cd.band_lo && band_hi <= cd.band_hi);
        if (!covers) cd.reset_residency();
    }
    if (cd.jobs_resident == 0) {
        cd.filtered = want_filter;
        cd.band_lo = band_lo;
        cd.band_hi = band_hi;
    }
    const size_t from = cd.jobs_resident, to = comp.jobs.size();
    if (from == to) return FORMA_STATUS_OK;
    if (to - from >= (1u << 30)) {
        set_error("too many inserts in one batch");
        return FORMA_STATUS_CAPACITY;
    }
    auto wanted = [&](const PendingInsert& p) { return !cd.filtered || !(p.y_min >= cd.band_hi || p.y_max <= cd.band_lo); };

    if (!cd.staged_valid || cd.staged_from != from || cd.staged_to != to || cd.staged_filtered != cd.filtered ||
        (cd.filtered && (cd.staged_lo != cd.band_lo || cd.staged_hi != cd.band_hi))) {
        // (Re)build the pinned staging copy of the flatten programs of the wanted jobs in [from, to).
        size_t n_jobs = 0, n_splines = 0, n_quads = 0, n_pts = 0, n_recs = 0, n_xfs = 0;
        bool rational = false;  // any weight != 1 in the batch: 48-byte QuadUp, else 36-byte QuadUpPoly
        for (size_t j = from; j < to; ++j) {
            if (!wanted(comp.jobs[j])) continue;
            const FlattenProgram& prog = comp.jobs[j].data->program();
            rational = rational || prog.rational;
            ++n_jobs;
            n_xfs += comp.jobs[j].has_xf ? 1u : 0u;
            n_splines += prog.splines.size();
            n_recs += prog.points.size();
            n_quads += prog.quads.size();
            n_pts += prog.n_points;
        }
        if ((uint64_t)cd.n_resident + n_pts >= (1ull << 32)) {
            set_error("too many points in the segment buffer");
            return FORMA_STATUS_CAPACITY;
        }
        FORMA_CUDA_TRY(cudaStreamSynchronize(stream));  // staging may still be in flight
        FORMA_CUDA_TRY(cd.h_splines.reserve(n_splines + 1));
        FORMA_CUDA_TRY(cd.h_points.reserve(n_recs + 1));
        FORMA_CUDA_TRY(cd.h_kinds.reserve(n_recs + 1));
        FORMA_CUDA_TRY(cd.h_quads.reserve(n_quads + 1));
        FORMA_CUDA_TRY(cd.h_jobs.reserve(n_jobs + 1));
        FORMA_CUDA_TRY(cd.h_xfs.reserve(n_xfs + 1));
        size_t ji = 0, si = 0, qi = 0, pi = 0, ri = 0, xi = 0;
        for (size_t j = from; j < to; ++j) {
            const PendingInsert& p = comp.jobs[j];
            if (!wanted(p)) continue;
            const FlattenProgram& prog = p.data->program();
            FlattenJob& job = cd.h_jobs.ptr[ji++];
            job.first_point = (uint32_t)pi;  // relative to the batch; the batch lands at the device's resident point count
            job.quad_base = (uint32_t)qi;
            job.spline_base = (uint32_t)(prog.splines.empty() ? ri : si);
            job.n_splines = (uint32_t)prog.splines.size();
            job.geom_id = p.geom_id;
            job.xf_index = 0;
            if (p.has_xf) {
                std::memcpy(cd.h_xfs.ptr[xi].xf, p.xf, sizeof(p.xf));
                job.xf_index = (uint32_t)++xi;
            }
            if (!prog.splines.empty())
                std::memcpy(cd.h_splines.ptr + si, prog.splines.data(), prog.splines.size() * sizeof(SplineRec));
            if (!prog.points.empty()) {
                std::memcpy(cd.h_points.ptr + ri, prog.points.data(), prog.points.size() * sizeof(PointRec));
                std::memcpy(cd.h_kinds.ptr + ri, prog.kinds.data(), prog.kinds.size());
                ri += prog.points.size();
            }
            if (rational) {
                for (size_t q = 0; q < prog.quads.size(); ++q) cd.h_quads.ptr[qi + q] = quad_upload(prog.quads[q]);
            } else {  // the pinned buffer is sized for QuadUp; the smaller records share it
                QuadUpPoly* poly = reinterpret_cast<QuadUpPoly*>(cd.h_quads.ptr);
                for (size_t q = 0; q < prog.quads.size(); ++q) {
                    const QuadRec& s = prog.quads[q];
                    QuadUpPoly& u = poly[qi + q];
                    for (int k = 0; k < 3; ++k) {
                        u.px[k] = s.px[k];
                        u.py[k] = s.py[k];
                    }
                    u.prev_curv = s.prev_curv;
                    u.total = s.total;
                    u.step = s.step;
                }
            }
            si += prog.splines.size();
            qi += prog.quads.size();
            pi += prog.n_points;
        }
        cd.staged_valid = true;
        cd.staged_from = from;
        cd.staged_to = to;
        cd.staged_filtered = cd.filtered;
        cd.staged_lo = cd.band_lo;
        cd.staged_hi = cd.band_hi;
        cd.staged_jobs = n_jobs;
        cd.staged_splines = n_splines;
        cd.staged_recs = n_recs;
        cd.staged_quads = n_quads;
        cd.staged_points = n_pts;
        cd.staged_xfs = n_xfs;
        cd.staged_rational = rational;
    }  // else: the same batch as last time (an evicted composition) is uploaded again from the same staging
    cd.jobs_resident = to;
    if (!cd.staged_jobs) return FORMA_STATUS_OK;
    const uint32_t n_after = cd.n_resident + (uint32_t)cd.staged_points;
    FORMA_CUDA_TRY(cd.d_x.reserve(n_after, true, stream));
    FORMA_CUDA_TRY(cd.d_y.reserve(n_after, true, stream));
    FORMA_CUDA_TRY(cd.d_gid.reserve(n_after, true, stream));
    const size_t quad_bytes = cd.staged_rational ? sizeof(QuadUp) : sizeof(QuadUpPoly);
    FORMA_CUDA_TRY(up_splines.reserve(cd.staged_splines + 1));
    FORMA_CUDA_TRY(up_points.reserve(cd.staged_recs + 1));
    FORMA_CUDA_TRY(up_kinds.reserve(cd.staged_recs + 1));
    FORMA_CUDA_TRY(up_quads.reserve(cd.staged_quads + 1));
    FORMA_CUDA_TRY(up_jobs.reserve(cd.staged_jobs));
    FORMA_CUDA_TRY(up_xfs.reserve(cd.staged_xfs + 1));
    // The quadratics go first: their expansion kernel runs on a side stream while the copy
    // engine keeps sending the other records.
    bool expanding = false;
    if (upload_after) FORMA_CUDA_TRY(cudaStreamWaitEvent(stream, upload_after, 0));
    if (cd.staged_quads) {
        FORMA_CUDA_TRY(up_quads_raw.reserve(cd.staged_quads + 1));
        FORMA_CUDA_TRY(cudaMemcpyAsync(up_quads_raw.ptr, cd.h_quads.ptr, cd.staged_quads * quad_bytes, cudaMemcpyHostToDevice,
                                       stream));
        if (!aux_stream) {
            FORMA_CUDA_TRY(cudaStreamCreateWithFlags(&aux_stream, cudaStreamNonBlocking));
            FORMA_CUDA_TRY(cudaEventCreateWithFlags(&aux_ev[0], cudaEventDisableTiming));
            FORMA_CUDA_TRY(cudaEventCreateWithFlags(&aux_ev[1], cudaEventDisableTiming));
        }
        FORMA_CUDA_TRY(cudaEventRecord(aux_ev[0], stream));
        FORMA_CUDA_TRY(cudaStreamWaitEvent(aux_stream, aux_ev[0], 0));
        if (cd.staged_rational)
            launch_quad_expand(up_quads_raw.ptr, up_quads.ptr, (uint32_t)cd.staged_quads, aux_stream);
        else
            launch_quad_expand_poly(reinterpret_cast<const QuadUpPoly*>(up_quads_raw.ptr), up_quads.ptr,
                                    (uint32_t)cd.staged_quads, aux_stream);
        FORMA_CUDA_TRY(cudaEventRecord(aux_ev[1], aux_stream));
        expanding = true;
        ++launches;
    }
    if (cd.staged_splines)
        FORMA_CUDA_TRY(cudaMemcpyAsync(up_splines.ptr, cd.h_splines.ptr, cd.staged_splines * sizeof(SplineRec),
                                       cudaMemcpyHostToDevice, stream));
    if (cd.staged_recs) {
        FORMA_CUDA_TRY(cudaMemcpyAsync(up_points.ptr, cd.h_points.ptr, cd.staged_recs * sizeof(PointRec), cudaMemcpyHostToDevice,
                                       stream));
        FORMA_CUDA_TRY(cudaMemcpyAsync(up_kinds.ptr, cd.h_kinds.ptr, cd.staged_recs, cudaMemcpyHostToDevice, stream));
    }
    FORMA_CUDA_TRY(cudaMemcpyAsync(up_jobs.ptr, cd.h_jobs.ptr, cd.staged_jobs * sizeof(FlattenJob), cudaMemcpyHostToDevice, stream));
    if (cd.staged_xfs)
        FORMA_CUDA_TRY(cudaMemcpyAsync(up_xfs.ptr, cd.h_xfs.ptr, cd.staged_xfs * sizeof(JobXf), cudaMemcpyHostToDevice, stream));
    if (upload_done_ev) FORMA_CUDA_TRY(cudaEventRecord(upload_done_ev, stream));
    h2d_bytes += cd.staged_splines * sizeof(SplineRec) + cd.staged_recs * (sizeof(PointRec) + 1) +
                 cd.staged_quads * quad_bytes + cd.staged_jobs * sizeof(FlattenJob) + cd.staged_xfs * sizeof(JobXf);
    if (expanding) FORMA_CUDA_TRY(cudaStreamWaitEvent(stream, aux_ev[1], 0));
    launch_flatten_eval(up_splines.ptr, up_points.ptr, up_kinds.ptr, up_quads.ptr, up_jobs.ptr, up_xfs.ptr, (uint32_t)cd.staged_jobs,
                        (uint32_t)cd.staged_points, cd.n_resident, cd.d_x.ptr, cd.d_y.ptr, cd.d_gid.ptr, stream);
    ++launches;
    FORMA_CUDA_TRY(cudaGetLastError());
    cd.n_resident = n_after;
    return FORMA_STATUS_OK;
}

// geom id -> layer slot, layer records, style table (segment.rs:141-149 does
// these look-ups per point). The pinned host copies are rebuilt when the
// composition changed and re-uploaded when they are not resident.
int Renderer::upload_tables(Composition& comp, int64_t cache_id) {
    comp.compact_geom();  // renumbers the geometry ids the tables are built from (no-op unless half of the points are dead)
    CompDevice& cd = comp.on(res_key);
    if (comp.tables_dirty || comp.tables_cache_id != cache_id) {
        FORMA_CUDA_TRY(cudaStreamSynchronize(stream));  // an upload from the pinned tables may still be in flight
        int st = rebuild_tables(comp, cache_id);
        if (st) return st;
    }
    if (cd.tables_version == comp.tables_version) return FORMA_STATUS_OK;
    return upload_tables_device(comp, cd);
}

// Host part: the pinned copies of the tables (no CUDA work besides pinned allocations). A
// caller that renders one composition on several devices runs it once before its workers start.
int Renderer::rebuild_tables(Composition& comp, int64_t cache_id) {
    {
        std::vector<StopRec> stops;
        std::vector<uint16_t> texels;
        std::unordered_map<const void*, uint32_t> tex_offsets;
        uint32_t max_order = 0;
        for (auto& kv : comp.layers) max_order = std::max(max_order, kv.first);
        uint32_t n_orders = comp.layers.empty() ? 0u : max_order + 1u;
        uint32_t n_geoms = comp.next_dense_id;
        FORMA_CUDA_TRY(comp.h_layers.reserve(comp.layers.size() + 1));
        FORMA_CUDA_TRY(comp.h_styles.reserve(comp.layers.size() + 1));
        FORMA_CUDA_TRY(comp.h_order_to_style.reserve(n_orders + 1));
        FORMA_CUDA_TRY(comp.h_geom_slot.reserve(n_geoms + 1));
        std::fill(comp.h_order_to_style.ptr, comp.h_order_to_style.ptr + n_orders, -1);
        std::fill(comp.h_geom_slot.ptr, comp.h_geom_slot.ptr + n_geoms, -1);
        uint32_t slot = 0, n_styles = 0;
        bool any_xf = false;
        FORMA_CUDA_TRY(comp.h_layer_bits.reserve(comp.layers.size() + 1));
        std::unordered_map<std::string, uint32_t> interned;
        std::vector<int32_t> order_to_slot(n_orders, -1);
        for (auto& kv : comp.layers) {
            const Layer& l = *kv.second;
            LayerRec& r = comp.h_layers.ptr[slot];
            r.order = kv.first;
            r.enabled = l.enabled ? 1u : 0u;
            r.has_xf = l.has_xf ? 1u : 0u;
            r.ux = l.xf[0]; r.uy = l.xf[1]; r.vx = l.xf[2]; r.vy = l.xf[3]; r.tx = l.xf[4]; r.ty = l.xf[5];
            comp.h_layer_bits.ptr[slot] = (kv.first & 0x1FFFFFu) | (r.enabled << 21);
            any_xf = any_xf || l.has_xf;
            StyleRec s = l.props.rec;
            s.stop_first = (uint32_t)stops.size();
            s.stop_count = (uint32_t)l.props.stops.size();
            stops.insert(stops.end(), l.props.stops.begin(), l.props.stops.end());
            if (s.fill_type == 2u && l.props.texels) {
                auto it = tex_offsets.find(l.props.texels.get());
                if (it == tex_offsets.end()) {
                    uint32_t off = (uint32_t)(texels.size() / 4);
                    texels.insert(texels.end(), l.props.texels->begin(), l.props.texels->end());
                    it = tex_offsets.emplace(l.props.texels.get(), off).first;
                }
                s.tex_first = it->second;
            }
            s.unchanged = 0u;
            // Styles are interned like the reference's props interner (composition/interner.rs):
            // solid fills that compare equal share one record (paris-30k: 66 records for 50 620
            // layers); gradients / textures keep one record per layer.
            uint32_t style_index = n_styles;
            if (s.fill_type == 0u && s.func == 0u) {
                std::string key(reinterpret_cast<const char*>(&s), offsetof(StyleRec, gradient_type));
                auto it = interned.find(key);
                if (it == interned.end()) interned.emplace(std::move(key), n_styles);
                else style_index = it->second;
            }
            if (style_index == n_styles) comp.h_styles.ptr[n_styles++] = s;
            comp.h_order_to_style.ptr[kv.first] = (int32_t)style_index;
            order_to_slot[kv.first] = (int32_t)slot;
            ++slot;
        }
        for (auto& kv : comp.geom_to_order) {
            if (kv.second < 0 || kv.first >= n_geoms || (uint64_t)kv.second >= n_orders) continue;
            comp.h_geom_slot.ptr[kv.first] = order_to_slot[kv.second];
        }
        comp.layers_in_order = true;
        {
            int64_t last = -1;
            for (const PendingInsert& job : comp.jobs) {
                if (job.geom_id >= n_geoms) continue;
                int32_t s = comp.h_geom_slot.ptr[job.geom_id];
                if (s < 0) continue;
                int64_t order = (int64_t)comp.h_layers.ptr[s].order;
                if (order < last) {
                    comp.layers_in_order = false;
                    break;
                }
                last = order;
            }
        }
        FORMA_CUDA_TRY(comp.h_stops.reserve(stops.size() + 1));
        FORMA_CUDA_TRY(comp.h_texels.reserve(texels.size() + 1));
        if (!stops.empty()) std::memcpy(comp.h_stops.ptr, stops.data(), stops.size() * sizeof(StopRec));
        if (!texels.empty()) std::memcpy(comp.h_texels.ptr, texels.data(), texels.size() * sizeof(uint16_t));
        comp.n_layer_recs = slot;
        comp.layers_have_xf = any_xf;
        comp.n_style_recs = n_styles;
        comp.n_stops = stops.size();
        comp.n_texels = texels.size();
        comp.n_geoms = n_geoms;
        comp.n_orders = n_orders;
        comp.tables_dirty = false;
        comp.tables_cache_id = cache_id;
        ++comp.tables_version;
    }
    return FORMA_STATUS_OK;
}

int Renderer::upload_tables_device(Composition& comp, CompDevice& cd) {
    auto up = [&](auto& dbuf, const auto& hbuf, size_t n) -> cudaError_t {
        cudaError_t e = dbuf.reserve(n + 1);
        if (e != cudaSuccess || n == 0) return e;
        h2d_bytes += n * sizeof(*hbuf.ptr);
        return cudaMemcpyAsync(dbuf.ptr, hbuf.ptr, n * sizeof(*hbuf.ptr), cudaMemcpyHostToDevice, stream);
    };
    // Layers without transforms (the common case) travel as 4 bytes each instead of 36.
    if (comp.layers_have_xf) FORMA_CUDA_TRY(up(cd.d_layers, comp.h_layers, comp.n_layer_recs));
    else FORMA_CUDA_TRY(up(cd.d_layer_bits, comp.h_layer_bits, comp.n_layer_recs));
    FORMA_CUDA_TRY(up(cd.d_styles, comp.h_styles, comp.n_style_recs));
    FORMA_CUDA_TRY(up(cd.d_stops, comp.h_stops, comp.n_stops));
    FORMA_CUDA_TRY(up(cd.d_texels, comp.h_texels, comp.n_texels));
    FORMA_CUDA_TRY(up(cd.d_order_to_style, comp.h_order_to_style, comp.n_orders));
    FORMA_CUDA_TRY(up(cd.d_geom_slot, comp.h_geom_slot, comp.n_geoms));
    // Gradient records of the styles (only when some style is a gradient: n_stops > 0).
    FORMA_CUDA_TRY(cd.d_grads.reserve(comp.n_style_recs + 1));
    if (comp.n_stops) {
        launch_grad_setup(cd.d_styles.ptr, cd.d_stops.ptr, (uint32_t)comp.n_style_recs, cd.d_grads.ptr, stream);
        ++launches;
    }
    cd.tables_version = comp.tables_version;
    return FORMA_STATUS_OK;
}

// Stages 1½ + 2: fills `segs` with the unsorted pixel segments.
int Renderer::rasterize(Composition& comp, uint32_t width, uint32_t height, float band_lo, float band_hi,
                        uint32_t* n_out) {
    RasterArgs& ra = last_raster;  // kept for forma_renderer_lines
    last_raster_valid = true;
    CompDevice& cd = comp.on(res_key);
    ra.x = cd.d_x.ptr;
    ra.y = cd.d_y.ptr;
    ra.gid = cd.d_gid.ptr;
    ra.n_points = cd.n_resident;
    ra.geom_slot = cd.d_geom_slot.ptr;
    ra.n_geoms = comp.n_geoms;
    ra.layers = comp.layers_have_xf ? cd.d_layers.ptr : nullptr;
    ra.layer_bits = cd.d_layer_bits.ptr;
    ra.width = (float)width;
    ra.height = (float)height;
    ra.band_lo = band_lo;
    ra.band_hi = band_hi;
    uint32_t nb = raster_num_blocks(ra.n_points);
    FORMA_CUDA_TRY(block_sums.reserve(nb + 1));
    launch_line_count(ra, block_sums.ptr, totals.ptr + 0, totals.ptr + 4, stream);
    launches += nb ? 2 : 0;
    uint32_t n = 0;
    // One read-back: segment count + the largest tile coordinates (totals[4..5]).
    FORMA_CUDA_TRY(cudaMemcpyAsync(pinned_totals, totals.ptr, 6 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    // The emit pass does not need the count, only room for its output: launch it
    // into the buffer of the previous frames before waiting for the read-back, so
    // that the GPU keeps working while the host wakes up. Segments beyond the
    // capacity are dropped and the pass is repeated below in that (rare) case.
    const size_t spec_cap = speculation_enabled() ? std::min<size_t>(segs.capacity, 0xFFFFFFFFu) : 0;
    const bool speculated = spec_cap > 1 && nb;
    FORMA_CUDA_TRY(ensure_count_event());
    FORMA_CUDA_TRY(cudaEventRecord(count_ev, stream));
    if (speculated) {
        if (timer.ok) FORMA_CUDA_TRY(cudaEventRecord(timer.ev[1], stream));  // end of line setup (count pass)
        launch_raster_emit(ra, block_sums.ptr, segs.ptr, (uint32_t)(spec_cap - 1), stream);
        ++launches;
    }
    FORMA_CUDA_TRY(cudaEventSynchronize(count_ev));  // the read-back only, not the speculative launch
    n = pinned_totals[0];
    {
        // Already ordered by layer: no layer digits (see Composition::layers_in_order).
        const bool skip_layer_digits = options().sort_full_key == 0;
        const uint64_t layer_bound = (comp.layers_in_order && skip_layer_digits) ? 0u : (comp.n_orders ? comp.n_orders - 1u : 0u);
        const uint64_t bound[3] = {layer_bound, pinned_totals[4], pinned_totals[5]};
        segment_plan = make_sort_plan(segment_key_layout(), bound);  // layer, tile_x, tile_y
    }
    *n_out = n;
    last_segments = n;
    if (n >= (1u << 30)) {
        set_error("%u pixel segments exceed the 2^30 limit of the sort's look-back counters", n);
        return FORMA_STATUS_CAPACITY;
    }
    FORMA_CUDA_TRY(segs.reserve(n + 1));
    FORMA_CUDA_TRY(segs_tmp.reserve(n + 1));
    if (!speculated || (size_t)n + 1 > spec_cap) {
        if (!speculated && timer.ok) FORMA_CUDA_TRY(cudaEventRecord(timer.ev[1], stream));  // end of line setup (count pass)
        launch_raster_emit(ra, block_sums.ptr, segs.ptr, n, stream);
        launches += nb ? 1 : 0;
    }
    FORMA_CUDA_TRY(cudaGetLastError());
    return FORMA_STATUS_OK;
}

// The upload half of render() on its own: tables + the geometry that the rows of `crop` need and
// that is not resident yet. render() then finds everything in place.
int Renderer::prefetch(Composition& comp, uint64_t width, uint64_t height, const forma_rect* crop) {
    FORMA_CUDA_TRY(cudaSetDevice(device));
    const int ts = ensure_timer();
    if (ts) return ts;
    const uint32_t tiles_y = (uint32_t)((height + 15u) / 16u);
    uint32_t ty_lo = 0, ty_hi = tiles_y;
    if (crop) {  // as in render()
        ty_lo = (uint32_t)std::min<uint64_t>(crop->vert_start / 16u, tiles_y);
        ty_hi = (uint32_t)std::min<uint64_t>((crop->vert_end + 15u) / 16u, tiles_y);
        if (ty_hi < ty_lo) ty_hi = ty_lo;
    }
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[0], stream));
    prefetched = true;
    if (upload_after) FORMA_CUDA_TRY(cudaStreamWaitEvent(stream, upload_after, 0));
    const float band_lo = (float)(ty_lo * 16u), band_hi = (float)std::min<uint64_t>((uint64_t)ty_hi * 16u, height);
    int st = upload_tables(comp, -1);
    if (st) return st;
    return flush_geometry(comp, band_lo, band_hi, ty_lo > 0u || ty_hi < tiles_y);
}

int Renderer::render(Composition& comp, uint8_t* buffer, bool buffer_on_device, uint64_t width, uint64_t stride,
                     uint64_t height, const uint32_t channels_in[4], const float clear[4], const forma_rect* crop,
                     LayerCache* cache, forma_timings* timings, uint32_t format) {
    if (format > kFormatRgba32f) {
        set_error("invalid output format %u", format);
        return FORMA_STATUS_INVALID;
    }
    const uint64_t bpp = format_bytes_per_pixel(format), elem = format_element_bytes(format);
    // LinearLayout::new asserts (layout/mod.rs:188-193) + consts.rs limits.
    if (!buffer || width == 0 || height == 0 || width * bpp > stride || width > FORMA_MAX_WIDTH || height > FORMA_MAX_HEIGHT) {
        set_error("invalid render target %llux%llu stride %llu", (unsigned long long)width, (unsigned long long)height,
                  (unsigned long long)stride);
        return FORMA_STATUS_INVALID;
    }
    if (stride % elem != 0 || reinterpret_cast<uintptr_t>(buffer) % elem != 0) {
        set_error("float frame: stride %llu and buffer address must be multiples of %llu bytes", (unsigned long long)stride,
                  (unsigned long long)elem);
        return FORMA_STATUS_INVALID;
    }
    FORMA_CUDA_TRY(cudaSetDevice(device));
    last_slices = 0;
    {
        const int ts = ensure_timer();
        if (ts) return ts;
    }

    PaintScene S{};
    for (int k = 0; k < 4; ++k) {
        uint32_t c = channels_in[k];
        if (c > 5u) {
            set_error("invalid channel %u", c);
            return FORMA_STATUS_INVALID;
        }
        if (clear[3] == 1.0f && c == FORMA_CHANNEL_ALPHA) c = FORMA_CHANNEL_ONE;  // renderer.rs:87-92
        S.channels[k] = c;
        S.clear[k] = clear[k];
    }
    S.width = (uint32_t)width;
    S.height = (uint32_t)height;
    S.stride = (uint32_t)stride;
    FrameOut frame_out;
    frame_out.format = format;
    S.tiles_x = (S.width + 15u) / 16u;
    S.tiles_y = (S.height + 15u) / 16u;
    S.tx_lo = 0; S.tx_hi = S.tiles_x; S.ty_lo = 0; S.ty_hi = S.tiles_y;
    if (crop) {  // Rect::new, renderer.rs:43-52
        S.tx_lo = (uint32_t)std::min<uint64_t>(crop->hor_start / 16u, S.tiles_x);
        S.tx_hi = (uint32_t)std::min<uint64_t>((crop->hor_end + 15u) / 16u, S.tiles_x);
        S.ty_lo = (uint32_t)std::min<uint64_t>(crop->vert_start / 16u, S.tiles_y);
        S.ty_hi = (uint32_t)std::min<uint64_t>((crop->vert_end + 15u) / 16u, S.tiles_y);
        if (S.tx_hi < S.tx_lo) S.tx_hi = S.tx_lo;
        if (S.ty_hi < S.ty_lo) S.ty_hi = S.ty_lo;
    }

    if (!prefetched) FORMA_CUDA_TRY(cudaEventRecord(timer.ev[0], stream));
    prefetched = false;
    // Lines entirely above / below the painted tile rows cannot reach a painted tile: they are
    // culled per line (rasterize), and whole inserts are left out of the device's segment
    // buffer when the band is narrower than the frame (flush_geometry).
    const float band_lo = (float)(S.ty_lo * 16u), band_hi = (float)std::min<uint64_t>((uint64_t)S.ty_hi * 16u, height);
    const bool band_is_partial = S.ty_lo > 0u || S.ty_hi < S.tiles_y;
    int st = upload_tables(comp, -1);
    if (st) return st;
    st = flush_geometry(comp, band_lo, band_hi, band_is_partial);
    if (st) return st;
    CompDevice& cd = comp.on(res_key);
    S.styles = cd.d_styles.ptr;
    S.order_to_style = cd.d_order_to_style.ptr;
    S.n_orders = comp.n_orders;
    S.stops = cd.d_stops.ptr;
    S.grads = cd.d_grads.ptr;
    S.texels = cd.d_texels.ptr;

    const bool pack_written = cache && !buffer_on_device;
    if (cache) {  // renderer.rs:94-110
        const size_t cache_tiles = (size_t)S.tiles_x * S.tiles_y;
        // A frame of another output format starts the cache over like a new size does: its
        // solid colours were compared at another precision.
        if (!cache->has_size || cache->width != width || cache->height != height || cache->format != format) {
            cache->has_size = true;
            cache->width = width;
            cache->height = height;
            cache->format = format;
            cache->clear();
        }
        FORMA_CUDA_TRY(cache->tiles.reserve(cache_tiles));
        if (cache->needs_reset) {
            FORMA_CUDA_TRY(cudaMemsetAsync(cache->tiles.ptr, 0, cache_tiles * sizeof(uint2), stream));
            cache->needs_reset = false;
        }
        S.cache_tiles = cache->tiles.ptr;
        if (format != kFormatRgba8) {  // read only where a tile's has-solid bit is set, i.e. after it was written
            FORMA_CUDA_TRY(cache->solid_wide.reserve(cache_tiles));
            frame_out.cache_solid_wide = cache->solid_wide.ptr;
        }
        S.clear_unchanged = cache->has_clear && cache->clear_color[0] == clear[0] && cache->clear_color[1] == clear[1] &&
                            cache->clear_color[2] == clear[2] && cache->clear_color[3] == clear[3];
        // Layer::is_unchanged(cache_id) per style slot (renderer.rs:144-157); the slots
        // follow the iteration order of upload_tables.
        FORMA_CUDA_TRY(h_unchanged.reserve(comp.n_orders + 1));
        FORMA_CUDA_TRY(d_unchanged.reserve(comp.n_orders + 1));
        size_t slot = comp.n_orders;  // one byte per layer order
        std::memset(h_unchanged.ptr, 0, slot);
        for (auto& kv : comp.layers)
            if (kv.first < comp.n_orders) h_unchanged.ptr[kv.first] = (uint8_t)((kv.second->unchanged_bits >> cache->id) & 1u);
        if (slot) {
            FORMA_CUDA_TRY(cudaMemcpyAsync(d_unchanged.ptr, h_unchanged.ptr, slot, cudaMemcpyHostToDevice, stream));
            h2d_bytes += slot;
        }
        S.unchanged = d_unchanged.ptr;
        if (pack_written) {
            FORMA_CUDA_TRY(written_list.reserve(cache_tiles));
            FORMA_CUDA_TRY(cudaMemsetAsync(totals.ptr + 6, 0, sizeof(uint32_t), stream));
            S.written_list = written_list.ptr;
            S.written_count = totals.ptr + 6;
        }
    }

    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[7], stream));
    uint32_t n = 0;
    st = rasterize(comp, S.width, S.height, band_lo, band_hi, &n);
    if (st) return st;

    // Stage 3: sort.
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[2], stream));
    const uint32_t prev_cells = last_cells, prev_gaps = last_gaps;  // of this renderer's previous frame
    last_cells = last_entries = 0;
    int timed_sort_passes = 0;
    if (n > 1) {
        FORMA_CUDA_TRY(sort_scratch.reserve(radix_scratch_bytes(n)));
        SortResult sr = launch_radix_sort(segs.ptr, segs_tmp.ptr, nullptr, nullptr, n, segment_plan, sort_scratch.ptr, stream,
                                          timer.sort_ev);
        launches += sr.launches;
        timed_sort_passes = sr.timed_passes;
        if (sr.in_tmp) swap_buffers(segs, segs_tmp);
        FORMA_CUDA_TRY(cudaGetLastError());
    }
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[3], stream));

    // Stage 4: cells -> carries -> entries -> paint.
    size_t n_tiles_total = (size_t)S.tiles_x * S.tiles_y;
    last_tiles_x = S.tiles_x;
    last_tiles_y = S.tiles_y;
    FORMA_CUDA_TRY(tile_range.reserve(n_tiles_total));
    FORMA_CUDA_TRY(heavy_tiles.reserve(n_tiles_total * kHeavyListClasses));
    // Heavy tiles first (longest-processing-time order): their lists + counts (totals[8..11]).
    uint32_t* const heavy_lists = options().paint_lpt ? heavy_tiles.ptr : nullptr;
    uint32_t* const heavy_counts = totals.ptr + 8;
    uint8_t* fb = buffer;
    if (!buffer_on_device) {
        FORMA_CUDA_TRY(framebuffer.reserve((size_t)stride * height));
        fb = framebuffer.ptr;
    }
    uint32_t paint_launches = 1;
    // Tables + paint + copy-back, once or (rarely) twice. fast = without count read-backs: the
    // tables of a frame are normally about as large as those of the frame before, so every
    // kernel is launched over bounds derived from the previous counts (+ 25 % + 4096) and reads
    // the real counts from device memory (DevCounts); the host looks at them only after the
    // frame's final synchronisation. A count above its bound (the kernels then did nothing,
    // the frame holds the clear colour) sends the frame through the known-count path below.
    uint32_t fast_cell_bound = 0, fast_gap_bound = 0;
    auto tables_and_paint = [&](const bool fast) -> int {
    uint32_t n_cells = 0, n_gaps = 0, n_entries = 0;
    DevCounts dc;
    if (n > 0 && fast) {
        const uint64_t shrink = options().test_fast_shrink ? 2u : 1u;
        const uint32_t cell_bound = fast_cell_bound =
            (uint32_t)std::min<uint64_t>(((uint64_t)prev_cells + prev_cells / 4u + 4096u) / shrink, n);
        const uint32_t gap_bound = fast_gap_bound =
            (uint32_t)std::min<uint64_t>(((uint64_t)prev_gaps + prev_gaps / 4u + 4096u) / shrink, 0x7FFFFFFFu);
        FORMA_CUDA_TRY(scan_state.reserve(std::max({cells_state_words(n), scan_state_words(n), scan_state_words(cell_bound)})));
        FORMA_CUDA_TRY(cell_start.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(cell_key.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(cell_cover.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(carry_in.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(carry_after.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(key2.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(key2_tmp.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(perm.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(perm_tmp.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(gap_count.reserve((size_t)cell_bound + 1));
        FORMA_CUDA_TRY(ekey_tmp.reserve((size_t)gap_bound + 1));
        FORMA_CUDA_TRY(eid_tmp.reserve((size_t)gap_bound + 1));
        FORMA_CUDA_TRY(gkey_tmp.reserve((size_t)gap_bound + 1));
        FORMA_CUDA_TRY(gid_tmp.reserve((size_t)gap_bound + 1));
        FORMA_CUDA_TRY(gap_carry.reserve((size_t)gap_bound + 1));
        const size_t entry_bound = (size_t)cell_bound + gap_bound;
        FORMA_CUDA_TRY(ekey.reserve(entry_bound));
        FORMA_CUDA_TRY(eid.reserve(entry_bound));
        FORMA_CUDA_TRY(eflags.reserve(entry_bound));
        FORMA_CUDA_TRY(recs.reserve(entry_bound));
        FORMA_CUDA_TRY(sort_scratch.reserve(std::max(radix_scratch_bytes(cell_bound), radix_scratch_bytes(gap_bound))));
        dc.cells = totals.ptr + 1;
        dc.gaps = totals.ptr + 2;
        dc.cell_bound = cell_bound;
        dc.gap_bound = gap_bound;
        // Cells beyond cell_bound + 1 are dropped by the pass; the count it leaves in totals[1] is the real one.
        launch_cells(S, segs.ptr, n, scan_state.ptr, cell_start.ptr, cell_bound + 1u, totals.ptr + 1, cell_key.ptr,
                     cell_cover.ptr, key2.ptr, perm.ptr, stream);
        launches += 2;
        {
            SortResult sr = launch_radix_sort(key2.ptr, key2_tmp.ptr, perm.ptr, perm_tmp.ptr, cell_bound, carry_sort_plan(S),
                                              sort_scratch.ptr, stream, nullptr, dc.cells);
            launches += sr.launches;
            if (sr.in_tmp) {
                swap_buffers(key2, key2_tmp);
                swap_buffers(perm, perm_tmp);
            }
        }
        launch_carry_scan(S, key2.ptr, perm.ptr, cell_cover.ptr, cell_bound, carry_in.ptr, carry_after.ptr, gap_count.ptr,
                          stream, dc);
        launch_scan_u32(gap_count.ptr, cell_bound, totals.ptr + 2, scan_state.ptr, stream, dc.cells);
        launch_gap_fill(S, key2.ptr, perm.ptr, cell_key.ptr, carry_after.ptr, gap_count.ptr, cell_bound, ekey_tmp.ptr,
                        eid_tmp.ptr, gap_carry.ptr, totals.ptr + 2, gap_bound, gap_bound, stream, dc);
        launches += 3;
        {
            SortResult sr = launch_radix_sort(ekey_tmp.ptr, gkey_tmp.ptr, eid_tmp.ptr, gid_tmp.ptr, gap_bound, gap_sort_plan(S),
                                              sort_scratch.ptr, stream, nullptr, dc.gaps);
            launches += sr.launches;
            if (sr.in_tmp) {
                swap_buffers(ekey_tmp, gkey_tmp);
                swap_buffers(eid_tmp, gid_tmp);
            }
        }
        launch_merge_entries(S, cell_key.ptr, cell_bound, ekey_tmp.ptr, eid_tmp.ptr, gap_bound, cell_start.ptr, carry_in.ptr,
                             gap_carry.ptr, ekey.ptr, recs.ptr, eflags.ptr, stream, dc);
        ++launches;
        n_entries = cell_bound + gap_bound;  // grid of the tile index pass
        // The counts travel to the host behind everything else of the frame.
        FORMA_CUDA_TRY(cudaMemcpyAsync(pinned_totals + 1, totals.ptr + 1, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    } else if (n > 0) {
        // Cells: one pass finds the cell heads, counts them and sums their covers. The count is
        // read back, but nothing waits for it: the pass runs into the buffers of the previous
        // frames (writes beyond their capacity are dropped) and is repeated below only if
        // those turn out too small.
        FORMA_CUDA_TRY(scan_state.reserve(std::max(cells_state_words(n), scan_state_words(n))));
        if (!cell_start.capacity) {  // first frame: a guess that usually holds (cells ~ segments / 20)
            const size_t guess = (size_t)n / 8u + 4096u;
            FORMA_CUDA_TRY(cell_start.reserve(guess));
            FORMA_CUDA_TRY(cell_key.reserve(guess));
            FORMA_CUDA_TRY(cell_cover.reserve(guess));
            FORMA_CUDA_TRY(key2.reserve(guess));
            FORMA_CUDA_TRY(perm.reserve(guess));
        }
        auto cells_capacity = [&] {
            return (uint32_t)std::min({cell_start.capacity, cell_key.capacity, cell_cover.capacity, key2.capacity, perm.capacity,
                                       (size_t)0xFFFFFFFFu});
        };
        uint32_t cell_cap = cells_capacity();
        launch_cells(S, segs.ptr, n, scan_state.ptr, cell_start.ptr, cell_cap, totals.ptr + 1, cell_key.ptr, cell_cover.ptr,
                     key2.ptr, perm.ptr, stream);
        launches += 2;
        FORMA_CUDA_TRY(cudaMemcpyAsync(pinned_totals + 1, totals.ptr + 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        FORMA_CUDA_TRY(cudaEventRecord(count_ev, stream));
        FORMA_CUDA_TRY(cudaEventSynchronize(count_ev));
        n_cells = pinned_totals[1];
        const bool cells_fit = (size_t)n_cells + 1 <= cell_cap;
        FORMA_CUDA_TRY(cell_start.reserve(n_cells + 1));
        FORMA_CUDA_TRY(cell_key.reserve(n_cells + 1));
        FORMA_CUDA_TRY(cell_cover.reserve(n_cells + 1));
        FORMA_CUDA_TRY(carry_in.reserve(n_cells));
        FORMA_CUDA_TRY(carry_after.reserve(n_cells));
        FORMA_CUDA_TRY(key2.reserve(n_cells + 1));
        FORMA_CUDA_TRY(key2_tmp.reserve(n_cells + 1));
        FORMA_CUDA_TRY(perm.reserve(n_cells + 1));
        FORMA_CUDA_TRY(perm_tmp.reserve(n_cells + 1));
        FORMA_CUDA_TRY(gap_count.reserve(n_cells));
        if (!cells_fit) {  // the buffers were too small: the pass dropped the overflow
            cell_cap = cells_capacity();
            launch_cells(S, segs.ptr, n, scan_state.ptr, cell_start.ptr, cell_cap, totals.ptr + 1, cell_key.ptr, cell_cover.ptr,
                         key2.ptr, perm.ptr, stream);
            launches += 2;
        }
        FORMA_CUDA_TRY(sort_scratch.reserve(radix_scratch_bytes(n_cells)));
        {
            SortResult sr = launch_radix_sort(key2.ptr, key2_tmp.ptr, perm.ptr, perm_tmp.ptr, n_cells, carry_sort_plan(S),
                                              sort_scratch.ptr, stream);
            launches += sr.launches;
            if (sr.in_tmp) {
                swap_buffers(key2, key2_tmp);
                swap_buffers(perm, perm_tmp);
            }
        }
        launch_carry_scan(S, key2.ptr, perm.ptr, cell_cover.ptr, n_cells, carry_in.ptr, carry_after.ptr, gap_count.ptr,
                          stream);
        // gap_count -> exclusive offsets, in place (gap_fill only needs the offsets).
        launch_scan_u32(gap_count.ptr, n_cells, totals.ptr + 2, scan_state.ptr, stream);
        launches += 2;
        // Same scheme for the number of carry-only entries: gap_fill runs ahead of the read-back.
        FORMA_CUDA_TRY(cudaMemcpyAsync(pinned_totals + 2, totals.ptr + 2, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
        FORMA_CUDA_TRY(cudaEventRecord(count_ev, stream));
        // The speculative output survives only if the reserve(n_gaps + 1) calls below do not
        // reallocate: one element of every buffer is kept back (the sort's slack slot).
        size_t gap_cap = 0;
        if (speculation_enabled()) {
            const size_t room = std::min({ekey_tmp.capacity, eid_tmp.capacity, gap_carry.capacity});
            gap_cap = std::min<size_t>(room ? room - 1u : 0u, (size_t)last_gaps * 2u + 4096u /* also the number of threads launched */);
            if (test_gap_cap_override() && gap_cap) gap_cap = std::min<size_t>(gap_cap, test_gap_cap_override());
        }
        if (gap_cap) {
            launch_gap_fill(S, key2.ptr, perm.ptr, cell_key.ptr, carry_after.ptr, gap_count.ptr, n_cells,
                            ekey_tmp.ptr, eid_tmp.ptr, gap_carry.ptr, totals.ptr + 2, (uint32_t)gap_cap, (uint32_t)gap_cap, stream);
            ++launches;
        }
        FORMA_CUDA_TRY(cudaEventSynchronize(count_ev));
        n_gaps = pinned_totals[2];
        last_gaps = n_gaps;
        n_entries = n_cells + n_gaps;
        last_cells = n_cells;
        last_entries = n_entries;
        FORMA_CUDA_TRY(ekey.reserve(n_entries));
        FORMA_CUDA_TRY(eid.reserve(n_entries));
        FORMA_CUDA_TRY(ekey_tmp.reserve(n_gaps + 1));  // carry-only entries: keys / ids + sort scratch
        FORMA_CUDA_TRY(eid_tmp.reserve(n_gaps + 1));
        FORMA_CUDA_TRY(gkey_tmp.reserve(n_gaps + 1));
        FORMA_CUDA_TRY(gid_tmp.reserve(n_gaps + 1));
        FORMA_CUDA_TRY(gap_carry.reserve(n_gaps + 1));
        FORMA_CUDA_TRY(eflags.reserve(n_entries));
        if (n_gaps) {
            FORMA_CUDA_TRY(sort_scratch.reserve(radix_scratch_bytes(n_gaps)));
            if (!gap_cap || n_gaps > gap_cap) {
                launch_gap_fill(S, key2.ptr, perm.ptr, cell_key.ptr, carry_after.ptr, gap_count.ptr, n_cells,
                                ekey_tmp.ptr, eid_tmp.ptr, gap_carry.ptr, totals.ptr + 2, n_gaps, n_gaps, stream);
                ++launches;
            }
            SortResult sr = launch_radix_sort(ekey_tmp.ptr, gkey_tmp.ptr, eid_tmp.ptr, gid_tmp.ptr, n_gaps, gap_sort_plan(S),
                                              sort_scratch.ptr, stream);
            launches += sr.launches;
            if (sr.in_tmp) {
                swap_buffers(ekey_tmp, gkey_tmp);
                swap_buffers(eid_tmp, gid_tmp);
            }
        }
        FORMA_CUDA_TRY(recs.reserve(n_entries));
        launch_merge_entries(S, cell_key.ptr, n_cells, ekey_tmp.ptr, eid_tmp.ptr, n_gaps, cell_start.ptr, carry_in.ptr,
                             gap_carry.ptr, ekey.ptr, recs.ptr, eflags.ptr, stream);
        ++launches;
    }
    launch_tile_index(S, ekey.ptr, n_entries, tile_range.ptr, heavy_lists, heavy_counts, stream, dc);
    launches += n_entries ? 1 : 0;
    row_costs_rows = 0;
    if (track_row_costs && n > 0) {
        FORMA_CUDA_TRY(d_row_costs.reserve(3u * S.tiles_y));  // per row: cost, pixel segments, entries
        FORMA_CUDA_TRY(h_row_costs.reserve(3u * S.tiles_y));
        launch_row_costs(tile_range.ptr, S.tiles_x, S.tiles_y, segs.ptr, n, d_row_costs.ptr, stream, d_row_costs.ptr + S.tiles_y);
        ++launches;
        FORMA_CUDA_TRY(cudaMemcpyAsync(h_row_costs.ptr, d_row_costs.ptr, 3u * S.tiles_y * sizeof(unsigned long long),
                                       cudaMemcpyDeviceToHost, stream));
        row_costs_rows = S.tiles_y;
    }
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[4], stream));
    // Host frame without a layer cache: paint in bands of tile rows, every band on its own
    // stream followed by the copy of its rows to the host buffer. The band kernels are
    // persistent (one CTA per resident slot), so the CTAs of band k + 1 start as the warps of
    // band k run dry: the kernels overlap at their tails, and the PCIe transfer of a band
    // overlaps the painting of the following ones.
    bool copied_in_bands = false;
    paint_launches = 1;
    const uint32_t paint_rows = S.ty_hi - S.ty_lo;
    if (!buffer_on_device && !cache && paint_rows >= (copy_bands_override ? 8u : 32u) && S.tx_hi > S.tx_lo && band_copies_enabled()) {
        if (!band_streams_ok) {
            for (auto& e : band_ev) FORMA_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            band_streams_ok = true;
        }
        const uint64_t x0 = (uint64_t)S.tx_lo * 16u, x1 = std::min<uint64_t>((uint64_t)S.tx_hi * 16u, width);
        const uint32_t kCopyBands = std::max(1u, std::min(copy_bands(), paint_rows / 8u));
        // One band: paint and copy on the render stream itself.
        while (kCopyBands > 1u && band_streams_made < kCopyBands) {
            FORMA_CUDA_TRY(cudaStreamCreateWithFlags(&band_stream[band_streams_made], cudaStreamNonBlocking));
            ++band_streams_made;
        }
        if (kCopyBands > 1u) FORMA_CUDA_TRY(cudaEventRecord(band_ev[kMaxCopyBands], stream));  // the tables are ready
        for (uint32_t k = 0; k < kCopyBands; ++k) {
            PaintScene Sb = S;
            Sb.ty_lo = S.ty_lo + paint_rows * k / kCopyBands;
            Sb.ty_hi = S.ty_lo + paint_rows * (k + 1u) / kCopyBands;
            cudaStream_t bs = kCopyBands > 1u ? band_stream[k] : stream;
            if (kCopyBands > 1u) FORMA_CUDA_TRY(cudaStreamWaitEvent(bs, band_ev[kMaxCopyBands], 0));
            launch_paint(Sb, segs.ptr, recs.ptr, tile_range.ptr, heavy_lists, heavy_counts, eflags.ptr, fb, totals.ptr + 16 + k, bs, frame_out);
            ++launches;
            const uint64_t y0 = (uint64_t)Sb.ty_lo * 16u, y1 = std::min<uint64_t>((uint64_t)Sb.ty_hi * 16u, height);
            if (x1 > x0 && y1 > y0) {
                if (x0 == 0 && x1 * bpp == stride)  // whole rows without padding: one contiguous copy
                    FORMA_CUDA_TRY(cudaMemcpyAsync(buffer + y0 * stride, fb + y0 * stride, (y1 - y0) * stride, cudaMemcpyDeviceToHost, bs));
                else
                    FORMA_CUDA_TRY(cudaMemcpy2DAsync(buffer + y0 * stride + x0 * bpp, stride, fb + y0 * stride + x0 * bpp, stride,
                                                     (x1 - x0) * bpp, y1 - y0, cudaMemcpyDeviceToHost, bs));
                d2h_bytes += (x1 - x0) * bpp * (y1 - y0);
            }
            if (kCopyBands > 1u) FORMA_CUDA_TRY(cudaEventRecord(band_ev[k], bs));
        }
        for (uint32_t k = 0; kCopyBands > 1u && k < kCopyBands; ++k) FORMA_CUDA_TRY(cudaStreamWaitEvent(stream, band_ev[k], 0));
        paint_launches = kCopyBands;
        copied_in_bands = true;
    } else {
        launch_paint(S, segs.ptr, recs.ptr, tile_range.ptr, heavy_lists, heavy_counts, eflags.ptr, fb, totals.ptr + 3, stream, frame_out);
        ++launches;
    }
    FORMA_CUDA_TRY(cudaGetLastError());
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[5], stream));

    last_written_tiles = 0;
    if (pack_written) {
        // With a layer cache only the tiles this frame wrote may touch the host
        // buffer (TileWriteOp::None leaves its bytes alone): pack them on the
        // device, copy count + ids + pixels, scatter on the host.
        const size_t tile_words = 64u * bpp;  // one packed tile: 256 pixels of bpp bytes, in u32 words
        FORMA_CUDA_TRY(packed_tiles.reserve((size_t)S.tiles_x * S.tiles_y * tile_words));
        launch_gather_tiles(S, format, fb, packed_tiles.ptr, stream);
        ++launches;
        uint32_t n_written = 0;
        st = read_total(6, &n_written);
        if (st) return st;
        last_written_tiles = n_written;
        if (n_written) {
            FORMA_CUDA_TRY(h_written_list.reserve(n_written));
            FORMA_CUDA_TRY(h_packed_tiles.reserve((size_t)n_written * tile_words));
            FORMA_CUDA_TRY(cudaMemcpyAsync(h_written_list.ptr, written_list.ptr, n_written * sizeof(uint32_t),
                                           cudaMemcpyDeviceToHost, stream));
            FORMA_CUDA_TRY(cudaMemcpyAsync(h_packed_tiles.ptr, packed_tiles.ptr, (size_t)n_written * tile_words * 4u,
                                           cudaMemcpyDeviceToHost, stream));
            FORMA_CUDA_TRY(cudaStreamSynchronize(stream));
            d2h_bytes += (uint64_t)n_written * (tile_words * 4u + 4u);
            if (format == kFormatRgba8) {
                for (uint32_t i = 0; i < n_written; ++i) {  // LinearLayout::write, layout/mod.rs:265-282
                    const uint32_t tile = h_written_list.ptr[i];
                    const uint64_t x0 = (uint64_t)(tile % S.tiles_x) * 16u, y0 = (uint64_t)(tile / S.tiles_x) * 16u;
                    const uint64_t cols = std::min<uint64_t>(16u, width - x0), rows = std::min<uint64_t>(16u, height - y0);
                    const uint32_t* src = h_packed_tiles.ptr + (size_t)i * 256u;
                    uint8_t* dst = buffer + y0 * stride + x0 * 4u;
                    if (cols == 16u) {  // whole tile rows: fixed-size copies the compiler turns into vector moves
                        for (uint64_t r = 0; r < rows; ++r) std::memcpy(dst + r * stride, src + r * 16u, 64);
                    } else {
                        for (uint64_t r = 0; r < rows; ++r) std::memcpy(dst + r * stride, src + r * 16u, cols * 4u);
                    }
                }
            } else {
                for (uint32_t i = 0; i < n_written; ++i) {
                    const uint32_t tile = h_written_list.ptr[i];
                    const uint64_t x0 = (uint64_t)(tile % S.tiles_x) * 16u, y0 = (uint64_t)(tile / S.tiles_x) * 16u;
                    const uint64_t cols = std::min<uint64_t>(16u, width - x0), rows = std::min<uint64_t>(16u, height - y0);
                    const uint8_t* src = reinterpret_cast<const uint8_t*>(h_packed_tiles.ptr + (size_t)i * tile_words);
                    uint8_t* dst = buffer + y0 * stride + x0 * bpp;
                    for (uint64_t r = 0; r < rows; ++r) std::memcpy(dst + r * stride, src + r * 16u * bpp, cols * bpp);
                }
            }
        }
    } else if (!buffer_on_device && !copied_in_bands) {
        // Only the cropped tile rectangle is written by the reference
        // (cpu/painter/mod.rs:524-529,589-593); padding bytes beyond width*bpp stay untouched.
        uint64_t x0 = (uint64_t)S.tx_lo * 16u, x1 = std::min<uint64_t>((uint64_t)S.tx_hi * 16u, width);
        uint64_t y0 = (uint64_t)S.ty_lo * 16u, y1 = std::min<uint64_t>((uint64_t)S.ty_hi * 16u, height);
        if (x1 > x0 && y1 > y0) {
            FORMA_CUDA_TRY(cudaMemcpy2DAsync(buffer + y0 * stride + x0 * bpp, stride, fb + y0 * stride + x0 * bpp, stride,
                                             (x1 - x0) * bpp, y1 - y0, cudaMemcpyDeviceToHost, stream));
            d2h_bytes += (x1 - x0) * bpp * (y1 - y0);
        }
    }
    FORMA_CUDA_TRY(cudaEventRecord(timer.ev[6], stream));
    FORMA_CUDA_TRY(cudaStreamSynchronize(stream));
    if (fast && n > 0) {
        last_cells = pinned_totals[1];
        last_gaps = pinned_totals[2];
        last_entries = last_cells + last_gaps;
    }
    return FORMA_STATUS_OK;
    };  // tables_and_paint
    // (pack_written: the host scatter of the written tiles must not see a frame that is redone.)
    bool fast = options().sync_free && n > 0 && prev_cells > 0 && !pack_written;
    st = tables_and_paint(fast);
    if (st) return st;
    last_tables_redone = false;
    if (fast && n > 0 && (last_cells > fast_cell_bound || last_gaps > fast_gap_bound)) {
        last_tables_redone = true;
        st = tables_and_paint(false);
        if (st) return st;
    }
    last_tables_sync_free = fast && !last_tables_redone;
    // The stage times are read from the events when somebody asks for them (resolve_times): a dozen
    // event queries are not part of rendering a frame.
    times_pending = true;
    pending_sort_passes = timed_sort_passes;
    pending_paint_launches = paint_launches;
    if (timings) resolve_times();
    if (timings) {
        timings->line_setup_ms = stage_ms[1];
        timings->rasterize_ms = stage_ms[2];
        timings->sort_ms = stage_ms[3];
        timings->paint_ms = stage_ms[4] + stage_ms[5];
        timings->n_lines = cd.n_resident ? cd.n_resident - 1 : 0;
        timings->n_segments = n;
    }
    if (cache) {  // renderer.rs:217-223
        cache->has_clear = true;
        std::memcpy(cache->clear_color, clear, sizeof(cache->clear_color));
        for (auto& kv : comp.layers) {
            if (kv.second->enabled) kv.second->unchanged_bits |= 1u << cache->id;
            else kv.second->unchanged_bits &= ~(1u << cache->id);
        }
    }
    return FORMA_STATUS_OK;
}

}  // namespace forma

// ===========================================================================
// C ABI
// ===========================================================================
using namespace forma;

struct forma_path_builder { PathBuilder b; };
struct forma_path { Path p; std::vector<float> x, y; std::vector<uint8_t> c; };
struct forma_composition { Composition c; };
struct forma_layer;  // == forma::Layer
struct forma_renderer_multi;
struct forma_renderer {
    Renderer r;
    // Host-frame pipeline (forma_renderer_render): slice renderers on this renderer's device,
    // created at the first frame that is sliced.
    forma_renderer_multi* slicer = nullptr;
    ~forma_renderer();
};
struct forma_layer_cache { LayerCache c; };

static Layer* L(forma_layer* l) { return reinterpret_cast<Layer*>(l); }
static forma_layer* H(Layer* l) { return reinterpret_cast<forma_layer*>(l); }

// No C++ exception crosses the C ABI: a failed host allocation (std::bad_alloc
// from the containers behind these calls) is reported through the call's error
// value and forma_last_error() like any other failure.
// Host-frame pipeline (defined next to the multi-device renderer): returns -1 when the frame is
// not sliced and the plain path has to render it.
static int sliced_host_render(forma_renderer* r, forma_composition* c, uint8_t* buffer, uint64_t width, uint64_t stride,
                              uint64_t height, const uint32_t channels[4], const float clear[4], const forma_rect* crop,
                              forma_timings* timings);

template <class R, class F>
static R guarded(R on_error, F&& f) noexcept {
    try {
        return f();
    } catch (const std::exception& e) {
        set_error("host error: %s", e.what());
    } catch (...) {
        set_error("host error: unknown exception");
    }
    return on_error;
}
template <class F>
static void guarded_void(F&& f) noexcept {
    guarded(0, [&] { f(); return 0; });
}

extern "C" {

const char* forma_last_error(void) { return g_error.c_str(); }

forma_path_builder* forma_path_builder_new(void) {
    return guarded((forma_path_builder*)nullptr, [] { return new forma_path_builder(); });
}
void forma_path_builder_free(forma_path_builder* pb) { delete pb; }
void forma_path_builder_move_to(forma_path_builder* pb, float x, float y) {
    guarded_void([&] { pb->b.move_to({x, y}); });
}
void forma_path_builder_line_to(forma_path_builder* pb, float x, float y) {
    guarded_void([&] { pb->b.line_to({x, y}); });
}
void forma_path_builder_quad_to(forma_path_builder* pb, float x1, float y1, float x2, float y2) {
    guarded_void([&] { pb->b.quad_to({x1, y1}, {x2, y2}); });
}
void forma_path_builder_cubic_to(forma_path_builder* pb, float x1, float y1, float x2, float y2, float x3, float y3) {
    guarded_void([&] { pb->b.cubic_to({x1, y1}, {x2, y2}, {x3, y3}); });
}
void forma_path_builder_rat_quad_to(forma_path_builder* pb, float x1, float y1, float x2, float y2, float w) {
    guarded_void([&] { pb->b.rat_quad_to({x1, y1}, {x2, y2}, w); });
}
void forma_path_builder_rat_cubic_to(forma_path_builder* pb, float x1, float y1, float x2, float y2, float x3,
                                     float y3, float w1, float w2) {
    guarded_void([&] { pb->b.rat_cubic_to({x1, y1}, {x2, y2}, {x3, y3}, w1, w2); });
}
forma_path* forma_path_builder_build(forma_path_builder* pb) {
    return guarded((forma_path*)nullptr, [&] {
        std::unique_ptr<forma_path> p(new forma_path());
        p->p = pb->b.build();
        return p.release();
    });
}
forma_path* forma_path_transform(const forma_path* src, const float m[9]) {
    return guarded((forma_path*)nullptr, [&] {
        std::unique_ptr<forma_path> p(new forma_path());
        p->p = src->p.transformed(m);
        return p.release();
    });
}
void forma_path_free(forma_path* p) { delete p; }

void forma_path_program_stats(forma_path* p, uint64_t out[6]) {
    const FlattenProgram& prog = p->p.data->program();
    out[0] = prog.n_points;
    out[1] = prog.quads.size();
    out[2] = prog.splines.size();
    out[3] = prog.points.size();
    out[4] = prog.rational ? 1 : 0;
    out[5] = prog.n_contour_ends;
}

// Evaluates the path's flatten program on the current device and copies the
// points back (inspection only; rendering never copies points to the host).
static int path_segments_impl(forma_path* p, const float** x, const float** y, const uint8_t** contour, uint64_t* n) {
    const FlattenProgram& prog = p->p.data->program();
    uint32_t count = prog.n_points;
    p->x.assign(count, 0.0f);
    p->y.assign(count, 0.0f);
    p->c.assign(count, 0);
    *n = count;
    *x = p->x.data();
    *y = p->y.data();
    *contour = p->c.data();
    if (!count) return FORMA_STATUS_OK;
    int dev_count = 0;
    if (cudaGetDeviceCount(&dev_count) != cudaSuccess || dev_count == 0) {
        set_error("forma_path_segments: no CUDA device (flatten evaluation has no CPU fallback)");
        return FORMA_STATUS_NO_DEVICE;
    }
    DeviceBuffer<SplineRec> dc;
    DeviceBuffer<QuadRec> dq;
    DeviceBuffer<FlattenJob> dj;
    DeviceBuffer<float> dx, dy;
    DeviceBuffer<uint32_t> dg;
    FORMA_CUDA_TRY(dc.reserve(prog.splines.size() + 1));
    FORMA_CUDA_TRY(dq.reserve(prog.quads.size() + 1));
    FORMA_CUDA_TRY(dj.reserve(1));
    FORMA_CUDA_TRY(dx.reserve(count));
    FORMA_CUDA_TRY(dy.reserve(count));
    FORMA_CUDA_TRY(dg.reserve(count));
    FlattenJob job{};
    job.first_point = 0;
    job.quad_base = 0;
    job.spline_base = 0;
    job.n_splines = (uint32_t)prog.splines.size();
    job.geom_id = 1;
    job.xf_index = p->p.has_xf ? 1u : 0u;
    JobXf job_xf{};
    std::memcpy(job_xf.xf, p->p.xf, sizeof(job_xf.xf));
    DeviceBuffer<JobXf> dxf;
    FORMA_CUDA_TRY(dxf.reserve(1));
    FORMA_CUDA_TRY(cudaMemcpy(dxf.ptr, &job_xf, sizeof(job_xf), cudaMemcpyHostToDevice));
    DeviceBuffer<PointRec> dp;
    DeviceBuffer<uint8_t> dk;
    FORMA_CUDA_TRY(dp.reserve(prog.points.size() + 1));
    FORMA_CUDA_TRY(dk.reserve(prog.kinds.size() + 1));
    if (!prog.splines.empty())
        FORMA_CUDA_TRY(cudaMemcpy(dc.ptr, prog.splines.data(), prog.splines.size() * sizeof(SplineRec), cudaMemcpyHostToDevice));
    if (!prog.points.empty()) {
        FORMA_CUDA_TRY(cudaMemcpy(dp.ptr, prog.points.data(), prog.points.size() * sizeof(PointRec), cudaMemcpyHostToDevice));
        FORMA_CUDA_TRY(cudaMemcpy(dk.ptr, prog.kinds.data(), prog.kinds.size(), cudaMemcpyHostToDevice));
    }
    if (!prog.quads.empty()) {  // same route as rendering: upload the control points, expand on the device
        std::vector<QuadUp> ups(prog.quads.size());
        for (size_t q = 0; q < ups.size(); ++q) ups[q] = quad_upload(prog.quads[q]);
        DeviceBuffer<QuadUp> du;
        FORMA_CUDA_TRY(du.reserve(ups.size()));
        FORMA_CUDA_TRY(cudaMemcpy(du.ptr, ups.data(), ups.size() * sizeof(QuadUp), cudaMemcpyHostToDevice));
        launch_quad_expand(du.ptr, dq.ptr, (uint32_t)ups.size(), 0);
        FORMA_CUDA_TRY(cudaDeviceSynchronize());
    }
    FORMA_CUDA_TRY(cudaMemcpy(dj.ptr, &job, sizeof(job), cudaMemcpyHostToDevice));
    launch_flatten_eval(dc.ptr, dp.ptr, dk.ptr, dq.ptr, dj.ptr, dxf.ptr, 1, count, 0, dx.ptr, dy.ptr, dg.ptr, 0);
    FORMA_CUDA_TRY(cudaGetLastError());
    FORMA_CUDA_TRY(cudaMemcpy(p->x.data(), dx.ptr, count * sizeof(float), cudaMemcpyDeviceToHost));
    FORMA_CUDA_TRY(cudaMemcpy(p->y.data(), dy.ptr, count * sizeof(float), cudaMemcpyDeviceToHost));
    for (const SplineRec& s : prog.splines) {  // the end point of a spline that ends a contour
        uint32_t end = s.first_point + ((s.info >> 30) & 1u) + (s.info & kSplineEvalMask);
        if ((s.info >> 31) && end < count) p->c[end] = 1;
    }
    for (size_t i = 0; i < prog.kinds.size() && i < count; ++i) p->c[i] = prog.kinds[i] == 1u;
    return FORMA_STATUS_OK;
}
int forma_path_segments(forma_path* p, const float** x, const float** y, const uint8_t** contour, uint64_t* n) {
    return guarded((int)FORMA_STATUS_CAPACITY, [&] { return path_segments_impl(p, x, y, contour, n); });
}

forma_composition* forma_composition_new(void) {
    return guarded((forma_composition*)nullptr, [] { return new forma_composition(); });
}
void forma_composition_free(forma_composition* c) { delete c; }
forma_layer* forma_composition_create_layer(forma_composition* c) {
    return guarded((forma_layer*)nullptr, [&] { return H(c->c.create_layer()); });
}
forma_layer* forma_composition_insert(forma_composition* c, uint32_t order, forma_layer* layer, int* status) {
    if (order > kLayerLimit) {
        if (status) *status = FORMA_ERR_ORDER_LIMIT;
        return nullptr;
    }
    if (status) *status = FORMA_OK;
    return guarded((forma_layer*)nullptr, [&] { return H(c->c.insert(order, L(layer))); });
}
forma_layer* forma_composition_remove(forma_composition* c, uint32_t order) {
    return guarded((forma_layer*)nullptr, [&] { return H(c->c.remove(order)); });
}
forma_layer* forma_composition_get(forma_composition* c, uint32_t order) { return H(c->c.get(order)); }
forma_layer* forma_composition_get_mut_or_insert_default(forma_composition* c, uint32_t order, int* status) {
    if (order > kLayerLimit) {
        if (status) *status = FORMA_ERR_ORDER_LIMIT;
        return nullptr;
    }
    if (status) *status = FORMA_OK;
    return guarded((forma_layer*)nullptr, [&] { return H(c->c.get_or_insert_default(order)); });
}
uint64_t forma_composition_len(forma_composition* c) { return c->c.layers.size(); }
void forma_layer_drop(forma_composition* c, forma_layer* l) {
    guarded_void([&] { c->c.drop(L(l)); });
}

uint64_t forma_layer_geom_id(forma_layer* l) { return L(l)->geom_id; }
int forma_layer_insert(forma_composition* c, forma_layer* l, forma_path* p) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        c->c.layer_insert(L(l), p->p);
        return (int)FORMA_OK;
    });
}
int forma_layer_clear(forma_composition* c, forma_layer* l) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        c->c.layer_clear(L(l));
        return (int)FORMA_OK;
    });
}
int forma_layer_set_is_enabled(forma_composition* c, forma_layer* l, int enabled) {
    L(l)->enabled = enabled != 0;
    c->c.mark_dirty();
    return FORMA_OK;
}
int forma_layer_is_enabled(forma_layer* l) { return L(l)->enabled ? 1 : 0; }

int forma_layer_set_transform(forma_composition* c, forma_layer* l, const float t[6]) {
    // AffineTransform::from([f32; 6]): ux = t0, vx = t1, uy = t2, vy = t3, tx = t4, ty = t5
    float ux = t[0], vx = t[1], uy = t[2], vy = t[3], tx = t[4], ty = t[5];
    if (!geom_pres_ok(ux, uy, vx, vy)) {
        set_error("GeomPresTransformError::ExceededScalingFactor");
        return FORMA_ERR_INVALID_ARGUMENT;
    }
    Layer* layer = L(l);
    bool has = !(ux == 1.0f && uy == 0.0f && vx == 0.0f && vy == 1.0f && tx == 0.0f && ty == 0.0f);
    float xf[6] = {ux, uy, vx, vy, tx, ty};
    bool same = has == layer->has_xf && (!has || std::memcmp(xf, layer->xf, sizeof(xf)) == 0 ||
                                         (xf[0] == layer->xf[0] && xf[1] == layer->xf[1] && xf[2] == layer->xf[2] &&
                                          xf[3] == layer->xf[3] && xf[4] == layer->xf[4] && xf[5] == layer->xf[5]));
    if (!same) {  // layer.rs:294-299
        layer->unchanged_bits = 0;
        layer->has_xf = has;
        std::memcpy(layer->xf, xf, sizeof(xf));
        c->c.mark_dirty();
    }
    return FORMA_OK;
}

// styling.rs:224-249 — forma's own f16 (no denormals, values in [0, 1]).
static uint16_t f16_from(float v) {
    if (v == 0.0f) return 0;
    uint32_t u;
    std::memcpy(&u, &v, 4);
    return (uint16_t)((u - 0x38000000u) >> 13);
}

static int layer_set_props_impl(forma_composition* c, forma_layer* l, const forma_props* p) {
    HostProps hp;
    StyleRec& s = hp.rec;
    s.fill_rule = p->fill_rule;
    s.func = p->func;
    s.clip_layers = p->clip_layers;
    s.is_clipped = p->is_clipped ? 1u : 0u;
    s.blend_mode = p->blend_mode;
    s.fill_type = p->fill_type;
    if (s.fill_rule > 1u || s.func > 1u || s.blend_mode > 15u || s.fill_type > 2u) {
        set_error("forma_layer_set_props: enum value out of range");
        return FORMA_ERR_INVALID_ARGUMENT;
    }
    s.color[0] = p->color.r; s.color[1] = p->color.g; s.color[2] = p->color.b; s.color[3] = p->color.a;
    if (s.func == FORMA_FUNC_DRAW && s.fill_type == FORMA_FILL_GRADIENT) {
        if (p->n_stops < 2 || !p->stops) {  // GradientBuilder::build -> None, styling.rs:107-109
            set_error("a gradient needs at least 2 stops");
            return FORMA_ERR_INVALID_ARGUMENT;
        }
        s.gradient_type = p->gradient_type;
        s.start[0] = p->start[0]; s.start[1] = p->start[1];
        s.end[0] = p->end[0]; s.end[1] = p->end[1];
        float incr = 1.0f / (float)(p->n_stops - 1);
        for (uint32_t i = 0; i < p->n_stops; ++i) {
            StopRec r;
            r.color[0] = p->stops[i].color.r; r.color[1] = p->stops[i].color.g;
            r.color[2] = p->stops[i].color.b; r.color[3] = p->stops[i].color.a;
            float stop = p->stops[i].stop;
            if (stop == -1.0f) stop = (float)i * incr;  // styling.rs:111-116
            else if (!(stop >= 0.0f && stop <= 1.0f)) {
                set_error("gradient stops must be between 0.0 and 1.0");
                return FORMA_ERR_INVALID_ARGUMENT;
            }
            r.stop = stop;
            hp.stops.push_back(r);
        }
    }
    if (s.func == FORMA_FUNC_DRAW && s.fill_type == FORMA_FILL_TEXTURE) {
        size_t n = (size_t)p->tex_width * p->tex_height;
        if (!n || !p->tex_linear_rgba) {
            set_error("empty texture");
            return FORMA_ERR_INVALID_ARGUMENT;
        }
        // Reuse the texel block when the same image is set again on this layer.
        auto tex = std::make_shared<std::vector<uint16_t>>(n * 4);
        for (size_t i = 0; i < n * 4; ++i) (*tex)[i] = f16_from(p->tex_linear_rgba[i]);
        Layer* layer = L(l);
        if (layer->props.texels && *layer->props.texels == *tex) tex = layer->props.texels;
        hp.texels = tex;
        for (int i = 0; i < 6; ++i) s.tex_xf[i] = p->tex_transform[i];
        s.tex_width = p->tex_width;
        s.tex_max_x = (float)p->tex_width - 1.0f;
        s.tex_max_y = (float)p->tex_height - 1.0f;
    }
    Layer* layer = L(l);
    if (!layer->props.equals(hp)) {  // layer.rs:341-348
        layer->unchanged_bits = 0;
        layer->props = std::move(hp);
        c->c.mark_dirty();
    }
    return FORMA_OK;
}
int forma_layer_set_props(forma_composition* c, forma_layer* l, const forma_props* p) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] { return layer_set_props_impl(c, l, p); });
}

static forma_renderer* renderer_new_impl(int device_ordinal) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("no CUDA device available (%s); forma_b200 has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return nullptr;
    }
    if (device_ordinal < 0 || device_ordinal >= count) {
        set_error("device ordinal %d out of range (0..%d)", device_ordinal, count - 1);
        return nullptr;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device_ordinal) != cudaSuccess || prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device_ordinal, prop.major, prop.minor);
        return nullptr;
    }
    if (cudaSetDevice(device_ordinal) != cudaSuccess) {
        set_error("cudaSetDevice(%d) failed", device_ordinal);
        return nullptr;
    }
    forma_renderer* r = new forma_renderer();
    r->r.device = device_ordinal;
    r->r.res_key = device_ordinal;
    if (cudaMallocHost(&r->r.pinned_totals, 16 * sizeof(uint32_t)) != cudaSuccess || r->r.totals.reserve(64) != cudaSuccess ||
        cudaMemset(r->r.totals.ptr, 0, r->r.totals.capacity * sizeof(uint32_t)) != cudaSuccess) {
        set_error("allocation of renderer state failed");
        delete r;
        return nullptr;
    }
    return r;
}
forma_renderer* forma_renderer_new(int device_ordinal) {
    return guarded((forma_renderer*)nullptr, [&] { return renderer_new_impl(device_ordinal); });
}
void forma_renderer_free(forma_renderer* r) { delete r; }

void forma_renderer_set_stream(forma_renderer* r, void* cuda_stream) { r->r.stream = (cudaStream_t)cuda_stream; }

forma_layer_cache* forma_layer_cache_new(forma_renderer* r) {
    for (uint8_t id = 0; id < 32; ++id)
        if (!((r->r.caches_in_use >> id) & 1u)) {
            forma_layer_cache* c = new (std::nothrow) forma_layer_cache();
            if (!c) {
                set_error("forma_layer_cache_new: out of host memory");
                return nullptr;
            }
            r->r.caches_in_use |= 1u << id;
            c->c.id = id;
            return c;
        }
    set_error("forma_layer_cache_new: all 32 cache ids of this renderer are in use");
    return nullptr;
}
void forma_layer_cache_free(forma_renderer* r, forma_layer_cache* c) {
    if (r) r->r.caches_in_use &= ~(1u << c->c.id);
    delete c;
}
void forma_layer_cache_clear(forma_layer_cache* c) {
    if (c) c->c.clear();
}

int forma_renderer_render(forma_renderer* r, forma_composition* c, uint8_t* buffer, uint64_t width, uint64_t stride,
                          uint64_t height, const uint32_t channels[4], const float clear[4], const forma_rect* crop,
                          forma_layer_cache* cache, forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        if (!cache) {
            const int st = sliced_host_render(r, c, buffer, width, stride, height, channels, clear, crop, timings);
            if (st >= 0) return st;
        }
        return r->r.render(c->c, buffer, false, width, stride, height, channels, clear, crop, cache ? &cache->c : nullptr,
                           timings);
    });
}
int forma_renderer_render_device(forma_renderer* r, forma_composition* c, uint8_t* device_buffer, uint64_t width,
                                 uint64_t stride, uint64_t height, const uint32_t channels[4], const float clear[4],
                                 const forma_rect* crop, forma_layer_cache* cache, forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return r->r.render(c->c, device_buffer, true, width, stride, height, channels, clear, crop,
                           cache ? &cache->c : nullptr, timings);
    });
}
// Float frames are not sliced (sliced_host_render): the slice pipeline is off by default and
// measured not to pay (DESIGN.md section 3), so it is left as it is for RGBA8.
int forma_renderer_render_format(forma_renderer* r, forma_composition* c, void* buffer, uint32_t format, uint64_t width,
                                 uint64_t stride, uint64_t height, const uint32_t channels[4], const float clear[4],
                                 const forma_rect* crop, forma_layer_cache* cache, forma_timings* timings) {
    if (format == FORMA_FORMAT_RGBA8)
        return forma_renderer_render(r, c, static_cast<uint8_t*>(buffer), width, stride, height, channels, clear, crop, cache, timings);
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return r->r.render(c->c, static_cast<uint8_t*>(buffer), false, width, stride, height, channels, clear, crop,
                           cache ? &cache->c : nullptr, timings, format);
    });
}
int forma_renderer_render_device_format(forma_renderer* r, forma_composition* c, void* device_buffer, uint32_t format,
                                        uint64_t width, uint64_t stride, uint64_t height, const uint32_t channels[4],
                                        const float clear[4], const forma_rect* crop, forma_layer_cache* cache,
                                        forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return r->r.render(c->c, static_cast<uint8_t*>(device_buffer), true, width, stride, height, channels, clear, crop,
                           cache ? &cache->c : nullptr, timings, format);
    });
}
// --- shared frames (multi-GPU, see include/forma_b200.h) -----------------------
static_assert(sizeof(cudaIpcMemHandle_t) == sizeof(forma_ipc_handle), "CUDA IPC handles are 64 bytes");
int forma_shared_frame_create(int device, uint64_t bytes, void** device_ptr, forma_ipc_handle* handle) {
    if (!device_ptr || !handle || !bytes) {
        set_error("forma_shared_frame_create: bad arguments");
        return FORMA_STATUS_INVALID;
    }
    FORMA_CUDA_TRY(cudaSetDevice(device));
    void* p = nullptr;
    FORMA_CUDA_TRY(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        set_error("cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
        return FORMA_STATUS_CUDA;
    }
    std::memcpy(handle->bytes, &h, sizeof(h));
    *device_ptr = p;
    return FORMA_STATUS_OK;
}
int forma_shared_frame_open(int device, const forma_ipc_handle* handle, void** device_ptr) {
    if (!device_ptr || !handle) {
        set_error("forma_shared_frame_open: bad arguments");
        return FORMA_STATUS_INVALID;
    }
    FORMA_CUDA_TRY(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle->bytes, sizeof(h));
    FORMA_CUDA_TRY(cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return FORMA_STATUS_OK;
}
int forma_shared_frame_close(int device, void* mapped_ptr) {
    FORMA_CUDA_TRY(cudaSetDevice(device));
    FORMA_CUDA_TRY(cudaIpcCloseMemHandle(mapped_ptr));
    return FORMA_STATUS_OK;
}
int forma_shared_frame_free(int device, void* device_ptr) {
    FORMA_CUDA_TRY(cudaSetDevice(device));
    FORMA_CUDA_TRY(cudaFree(device_ptr));
    return FORMA_STATUS_OK;
}

// ---------------------------------------------------------------------------
// Several GPUs behind one renderer (single process): tile-row bands, one worker thread and
// one forma_renderer per device. Every device makes the geometry of its band resident
// (flush_geometry's band filter), rasterizes, sorts and paints its band, and either copies
// the band's rows to the caller's host buffer or stores them into the frame in the first
// device's memory over NVLink (peer access). No collective: the bands are disjoint row
// ranges of one frame. The bands of the next frame are balanced on this frame's row costs.
// ---------------------------------------------------------------------------
}  // extern "C"

// Persistent worker threads of a multi-device (or sliced) renderer: run(n, f) executes f(0) on
// the calling thread and f(1) ... f(n - 1) on workers that live as long as the pool, so a frame
// of a millisecond does not pay for thread creation.
class WorkerPool {
   public:
    ~WorkerPool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv_work.notify_all();
        for (std::thread& t : threads) t.join();
    }
    void run(size_t n, const std::function<void(size_t)>& f) {
        if (n == 0) return;
        while (threads.size() + 1 < n) {
            const size_t index = threads.size() + 1;
            uint64_t seen;
            {
                std::lock_guard<std::mutex> lk(mu);
                seen = generation;
            }
            threads.emplace_back([this, index, seen] { worker(index, seen); });
        }
        if (n > 1) {
            std::lock_guard<std::mutex> lk(mu);
            job = &f;
            active = n;
            pending = threads.size();
            ++generation;
        }
        if (n > 1) cv_work.notify_all();
        f(0);
        if (n > 1) {
            std::unique_lock<std::mutex> lk(mu);
            cv_done.wait(lk, [&] { return pending == 0; });
            job = nullptr;
        }
    }

   private:
    void worker(size_t index, uint64_t seen) {
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv_work.wait(lk, [&] { return stop || generation != seen; });
            if (stop) return;
            seen = generation;
            const std::function<void(size_t)>* f = job;
            const size_t n = active;
            lk.unlock();
            if (index < n && f) {
                try {
                    (*f)(index);
                } catch (...) {  // jobs report through their own status words
                }
            }
            lk.lock();
            if (--pending == 0) cv_done.notify_one();
        }
    }
    std::vector<std::thread> threads;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    const std::function<void(size_t)>* job = nullptr;
    size_t active = 0, pending = 0;
    uint64_t generation = 0;
    bool stop = false;
};

struct forma_renderer_multi {
    std::vector<forma_renderer*> dev;
    std::vector<uint32_t> bounds;  // tile rows: band i = [bounds[i], bounds[i + 1])
    uint32_t bounds_lo = 0, bounds_hi = 0;
    bool peer_ok = true;           // every device may store into the first device's memory
    std::vector<double> last_ms;   // device-timeline ms of each band in the last frame
    size_t active = 0;             // bands used by the last frame (a sliced host frame may use fewer than dev.size())
    uint64_t last_own_segments = 0, last_own_entries = 0;  // pixel segments / entries of the last frame, every band counting its own rows only
    WorkerPool pool;
};

static int multi_render_impl(forma_renderer_multi* m, forma_composition* c, uint8_t* buffer, bool on_device, uint64_t width,
                             uint64_t stride, uint64_t height, const uint32_t channels[4], const float clear[4],
                             const forma_rect* crop, forma_timings* timings, uint32_t format = kFormatRgba8, size_t n_use = 0,
                             bool chained_uploads = false) {
    const size_t n = n_use ? std::min(n_use, m->dev.size()) : m->dev.size();
    m->active = n;
    if (!n || !width || !height || width > FORMA_MAX_WIDTH || height > FORMA_MAX_HEIGHT) {
        set_error("forma_renderer_multi_render: invalid arguments");
        return FORMA_STATUS_INVALID;
    }
    if (on_device && n > 1 && !m->peer_ok) {
        set_error("forma_renderer_multi_render_device: peer access to the first device is not available");
        return FORMA_STATUS_INVALID;
    }
    Composition& comp = c->c;
    // Tile rows to paint (crop is tile-granular like cpu/renderer.rs:43-52).
    const uint32_t tiles_y = (uint32_t)((height + 15u) / 16u);
    uint32_t row_lo = 0, row_hi = tiles_y;
    forma_rect full{0, width, 0, height};
    if (crop) {
        full = *crop;
        row_lo = (uint32_t)std::min<uint64_t>(crop->vert_start / 16u, tiles_y);
        row_hi = (uint32_t)std::min<uint64_t>((crop->vert_end + 15u) / 16u, tiles_y);
        if (row_hi < row_lo) row_hi = row_lo;
    }
    if (m->bounds.size() != n + 1 || m->bounds_lo != row_lo || m->bounds_hi != row_hi) {  // first frame / new target: equal bands
        m->bounds.assign(n + 1, row_lo);
        for (size_t i = 0; i <= n; ++i) m->bounds[i] = row_lo + (uint32_t)(((uint64_t)(row_hi - row_lo) * i) / n);
        m->bounds_lo = row_lo;
        m->bounds_hi = row_hi;
    }
    // Host-side preparation, once: compaction, the pinned tables, the per-device records.
    comp.compact_geom();
    if (comp.tables_dirty || comp.tables_cache_id != -1) {
        for (forma_renderer* r : m->dev) {
            FORMA_CUDA_TRY(cudaSetDevice(r->r.device));
            FORMA_CUDA_TRY(cudaStreamSynchronize(r->r.stream));
        }
        int st = Renderer::rebuild_tables(comp, -1);
        if (st) return st;
    }
    for (forma_renderer* r : m->dev) comp.on(r->r.res_key);  // the workers only look their records up

    std::vector<int> status(n, FORMA_STATUS_OK);
    std::vector<std::string> errors(n);
    std::vector<forma_timings> tms(n);
    std::vector<std::vector<uint64_t>> costs(n);
    std::vector<uint64_t> own_segments(n, 0), own_entries(n, 0);
    m->last_ms.assign(n, 0.0);
    auto band_of = [&](size_t i, forma_rect* band) {
        const uint32_t r0 = m->bounds[i], r1 = m->bounds[i + 1];
        if (r1 <= r0) return false;
        *band = full;
        band->vert_start = std::max<uint64_t>(full.vert_start, (uint64_t)r0 * 16u);
        band->vert_end = std::min<uint64_t>(std::min<uint64_t>(full.vert_end, height), (uint64_t)r1 * 16u);
        return band->vert_end > band->vert_start;
    };
    if (chained_uploads) {
        // Slices of one device share its PCIe link: their uploads are issued here, in slice order,
        // each waiting for the one before (Renderer::upload_after), instead of all at once.
        for (size_t i = 0; i < n; ++i) {
            forma_rect band;
            if (!band_of(i, &band)) continue;
            const int st = m->dev[i]->r.prefetch(comp, width, height, &band);
            if (st) {
                for (size_t k = 0; k < n; ++k) m->dev[k]->r.prefetched = false;
                return st;
            }
        }
    }
    auto work = [&](size_t i) {
        const uint32_t r0 = m->bounds[i], r1 = m->bounds[i + 1];
        std::memset(&tms[i], 0, sizeof(forma_timings));
        forma_rect band;
        if (!band_of(i, &band)) return;
        Renderer& R = m->dev[i]->r;
        status[i] = guarded((int)FORMA_ERR_CAPACITY, [&] {
            return R.render(comp, buffer, on_device, width, stride, height, channels, clear, &band, nullptr, &tms[i], format);
        });
        if (status[i]) {
            errors[i] = forma_last_error();
            return;
        }
        m->last_ms[i] = R.stage_ms[7];
        costs[i].assign(tiles_y, 0);  // the frame's row costs came back behind the frame (track_row_costs)
        for (uint32_t r = 0; r < std::min(R.row_costs_rows, tiles_y); ++r) costs[i][r] = R.h_row_costs.ptr[r];
        // A line that crosses a band boundary is rasterized by both neighbours: the frame's
        // segment count is the sum of the segments every band has in its own rows.
        if (R.row_costs_rows == tiles_y) {
            uint64_t own = 0, own_e = 0;
            for (uint32_t r = r0; r < std::min(r1, tiles_y); ++r) {
                own += R.h_row_costs.ptr[tiles_y + r];
                own_e += R.h_row_costs.ptr[2u * tiles_y + r];
            }
            own_segments[i] = own;
            own_entries[i] = own_e;
        } else {
            own_segments[i] = R.last_segments;
            own_entries[i] = R.last_entries;
        }
    };
    m->pool.run(n, [&](size_t i) {
        try {
            work(i);
        } catch (const std::exception& e) {
            status[i] = FORMA_STATUS_CAPACITY;
            errors[i] = e.what();
        }
    });
    for (size_t i = 0; i < n; ++i)
        if (status[i]) {
            set_error("device %d: %s", m->dev[i]->r.device, errors[i].c_str());
            return status[i];
        }
    if (timings) {
        std::memset(timings, 0, sizeof(*timings));
        for (size_t i = 0; i < n; ++i) {  // stages: the slowest band; sizes: the whole frame
            timings->line_setup_ms = std::max(timings->line_setup_ms, tms[i].line_setup_ms);
            timings->rasterize_ms = std::max(timings->rasterize_ms, tms[i].rasterize_ms);
            timings->sort_ms = std::max(timings->sort_ms, tms[i].sort_ms);
            timings->paint_ms = std::max(timings->paint_ms, tms[i].paint_ms);
            timings->n_lines += tms[i].n_lines;
            timings->n_segments += own_segments[i];
        }
    }
    m->last_own_segments = m->last_own_entries = 0;
    for (size_t i = 0; i < n; ++i) {
        m->last_own_segments += own_segments[i];
        m->last_own_entries += own_entries[i];
    }
    // Next frame's bands: equal shares of this frame's row costs (+ a floor per row: every
    // tile is at least cleared and stored).
    if (n > 1 && row_hi > row_lo) {
        std::vector<double> cost(tiles_y, 0.0);
        const double floor_cost = 2.0 * (double)((width + 15u) / 16u);
        for (size_t i = 0; i < n; ++i)
            for (uint32_t r = m->bounds[i]; r < m->bounds[i + 1] && r < (uint32_t)costs[i].size(); ++r)
                cost[r] = (double)costs[i][r];
        double total = 0.0;
        for (uint32_t r = row_lo; r < row_hi; ++r) total += (cost[r] += floor_cost);
        // Bands that are still within 8 % of an equal share stay as they are: moving a boundary
        // makes the devices on both sides re-stage and re-upload their geometry.
        double worst = 0.0;
        for (size_t i = 0; i < n; ++i) {
            double band = 0.0;
            for (uint32_t r = m->bounds[i]; r < m->bounds[i + 1]; ++r) band += cost[r];
            worst = std::max(worst, band);
        }
        if (worst * (double)n <= 1.08 * total) return FORMA_STATUS_OK;
        std::vector<uint32_t> nb(1, row_lo);
        double run = 0.0;
        size_t k = 1;
        for (uint32_t r = row_lo; r < row_hi; ++r) {
            while (k < n && run + 0.5 * cost[r] >= total * (double)k / (double)n) {
                nb.push_back(r);
                ++k;
            }
            run += cost[r];
        }
        while (nb.size() < n) nb.push_back(row_hi);
        nb.push_back(row_hi);
        m->bounds = nb;
    }
    return FORMA_STATUS_OK;
}

extern "C" {

forma_renderer_multi* forma_renderer_multi_new(const int* devices, int n) {
    return guarded((forma_renderer_multi*)nullptr, [&]() -> forma_renderer_multi* {
        if (!devices || n < 1 || n > 64) {
            set_error("forma_renderer_multi_new: need 1..64 device ordinals");
            return nullptr;
        }
        std::unique_ptr<forma_renderer_multi> m(new forma_renderer_multi());
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j < i; ++j)
                if (devices[j] == devices[i]) {
                    set_error("forma_renderer_multi_new: device %d listed twice", devices[i]);
                    for (forma_renderer* r : m->dev) forma_renderer_free(r);
                    return nullptr;
                }
            forma_renderer* r = forma_renderer_new(devices[i]);
            if (!r) {
                for (forma_renderer* q : m->dev) forma_renderer_free(q);
                return nullptr;
            }
            // Each device renders on its own (non-blocking) stream.
            cudaStream_t st = nullptr;
            if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess) {
                r->r.stream = st;
                r->r.owns_stream = true;
            }
            r->r.track_row_costs = true;
            m->dev.push_back(r);
        }
        for (int i = 1; i < n; ++i) {  // stores into the first device's frame go over NVLink
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devices[i], devices[0]) != cudaSuccess || !can) {
                m->peer_ok = false;
                continue;
            }
            cudaSetDevice(devices[i]);
            cudaError_t e = cudaDeviceEnablePeerAccess(devices[0], 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) m->peer_ok = false;
            cudaGetLastError();
        }
        return m.release();
    });
}
void forma_renderer_multi_free(forma_renderer_multi* m) {
    if (!m) return;
    for (forma_renderer* r : m->dev) forma_renderer_free(r);
    delete m;
}
}  // extern "C"

forma_renderer::~forma_renderer() {
    if (slicer) forma_renderer_multi_free(slicer);
}

// Host frames as a pipeline of tile-row slices. A host frame is upload (the geometry that is not
// resident) -> line setup / rasterize / sort / tables -> paint -> copy-back; on one stream the
// copy engines idle while the SMs work and the other way round, and PCIe carries one direction
// at a time. Here the frame is cut into `host_slices` bands of tile rows; every slice is a
// renderer of its own on this device (own stream, own scratch, own residency record with the
// band filter of the multi-GPU path, so it uploads and evaluates only the geometry that can
// reach its rows) driven by its own host thread: slice k + 1 uploads while slice k computes
// and slice k - 1 copies back, and the two PCIe directions run at the same time. The slices are
// balanced on the previous frame's row costs like the bands of a multi-GPU frame. Results are
// those of a band render (tests/test_gpu_bench_scale.py: bands == whole frame).
// Not sliced: frames with a layer cache (the cache records belong to one renderer), layers with
// transforms (no band filter: every slice would upload everything), small compositions, short frames.
static int sliced_host_render(forma_renderer* r, forma_composition* c, uint8_t* buffer, uint64_t width, uint64_t stride,
                              uint64_t height, const uint32_t channels[4], const float clear[4], const forma_rect* crop,
                              forma_timings* timings) {
    Renderer& P = r->r;
    const int want = options().host_slices;
    if (want < 2 || !buffer || !width || !height || width > FORMA_MAX_WIDTH || height > FORMA_MAX_HEIGHT || width * 4 > stride)
        return -1;  // (invalid targets are reported by the plain path)
    for (int k = 0; k < 4; ++k)
        if (channels[k] > 5u) return -1;
    Composition& comp = c->c;
    if ((uint64_t)comp.n_points < (uint64_t)std::max(options().slice_min_points, 0)) return -1;
    const uint32_t tiles_y = (uint32_t)((height + 15u) / 16u);
    uint32_t row_lo = 0, row_hi = tiles_y;
    if (crop) {
        row_lo = (uint32_t)std::min<uint64_t>(crop->vert_start / 16u, tiles_y);
        row_hi = (uint32_t)std::min<uint64_t>((crop->vert_end + 15u) / 16u, tiles_y);
        if (crop->hor_end <= crop->hor_start) return -1;
    }
    if (row_hi <= row_lo) return -1;
    const size_t n = std::min<size_t>((size_t)want, (row_hi - row_lo) / 16u);  // at least 16 tile rows per slice
    if (n < 2) return -1;
    if (cudaSetDevice(P.device) != cudaSuccess) return -1;
    // The tables are rebuilt here (the slices find them clean) so that layers_have_xf is known.
    comp.compact_geom();
    if (comp.tables_dirty || comp.tables_cache_id != -1) {
        FORMA_CUDA_TRY(cudaStreamSynchronize(P.stream));
        if (r->slicer)
            for (forma_renderer* q : r->slicer->dev) FORMA_CUDA_TRY(cudaStreamSynchronize(q->r.stream));
        const int st = Renderer::rebuild_tables(comp, -1);
        if (st) return st;
    }
    if (comp.layers_have_xf) return -1;
    if (!r->slicer || r->slicer->dev.size() < n) {
        if (r->slicer) forma_renderer_multi_free(r->slicer);
        r->slicer = nullptr;
        std::unique_ptr<forma_renderer_multi> m(new forma_renderer_multi());
        for (size_t i = 0; i < (size_t)want; ++i) {
            forma_renderer* q = forma_renderer_new(P.device);
            if (!q) {
                for (forma_renderer* x : m->dev) forma_renderer_free(x);
                return FORMA_STATUS_CUDA;
            }
            cudaStream_t st = nullptr;
            if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
                forma_renderer_free(q);
                for (forma_renderer* x : m->dev) forma_renderer_free(x);
                set_error("sliced host frame: cannot create a stream");
                return FORMA_STATUS_CUDA;
            }
            q->r.stream = st;
            q->r.owns_stream = true;
            q->r.res_key = P.device + 4096 * (int)(i + 1);
            q->r.track_row_costs = true;
            if (cudaEventCreateWithFlags(&q->r.upload_done_ev, cudaEventDisableTiming) != cudaSuccess) q->r.upload_done_ev = nullptr;
            if (i > 0) q->r.upload_after = m->dev[i - 1]->r.upload_done_ev;
            m->dev.push_back(q);
        }
        r->slicer = m.release();
    }
    forma_renderer_multi* m = r->slicer;
    // The slices start behind whatever the caller has queued on this renderer's stream.
    if (!P.count_ev) FORMA_CUDA_TRY(P.ensure_count_event());
    FORMA_CUDA_TRY(cudaEventRecord(P.count_ev, P.stream));
    struct Before { uint64_t launches, h2d, d2h; };
    std::vector<Before> before(n);
    for (size_t i = 0; i < n; ++i) {
        Renderer& Q = m->dev[i]->r;
        Q.copy_bands_override = std::max(options().slice_bands, 1);
        FORMA_CUDA_TRY(cudaStreamWaitEvent(Q.stream, P.count_ev, 0));
        before[i] = {Q.launches, Q.h2d_bytes, Q.d2h_bytes};
    }
    const int st = multi_render_impl(m, c, buffer, false, width, stride, height, channels, clear, crop, timings, kFormatRgba8, n,
                                     options().slice_chain != 0);
    if (st) return st;
    // What the caller reads from this renderer after a frame: sums over the slices; stage times:
    // the slowest slice (the slices overlap, so their sum means nothing).
    P.last_segments = P.last_cells = P.last_entries = 0;
    for (double& v : P.stage_ms) v = 0.0;
    bool redone = false, all_fast = true;
    for (size_t i = 0; i < n; ++i) {
        const Renderer& Q = m->dev[i]->r;
        P.launches += Q.launches - before[i].launches;
        P.h2d_bytes += Q.h2d_bytes - before[i].h2d;
        P.d2h_bytes += Q.d2h_bytes - before[i].d2h;
        P.last_cells += Q.last_cells;
        for (int k = 0; k < 8; ++k) P.stage_ms[k] = std::max(P.stage_ms[k], Q.stage_ms[k]);
        redone = redone || Q.last_tables_redone;
        all_fast = all_fast && Q.last_tables_sync_free;
    }
    for (int k = 0; k < 4; ++k) {
        P.kernel_ms[k] = 0.0;
        P.kernel_launches[k] = 0;
    }
    P.last_tables_redone = redone;
    P.last_tables_sync_free = all_fast && !redone;
    P.times_pending = false;      // stage_ms was just set from the slices
    P.last_raster_valid = false;  // forma_renderer_lines describes the last unsliced render only
    P.last_written_tiles = 0;
    P.last_tiles_x = P.last_tiles_y = 0;
    P.last_segments = (uint32_t)std::min<uint64_t>(m->last_own_segments, 0xFFFFFFFFu);
    P.last_entries = (uint32_t)std::min<uint64_t>(m->last_own_entries, 0xFFFFFFFFu);
    // (cells: a slice also forms the cells of segments that boundary-crossing lines leave in its
    // neighbours' rows, so the sum over the slices is an upper bound of the frame's cell count)
    P.last_slices = (uint32_t)n;
    return FORMA_STATUS_OK;
}

extern "C" {

/* Slices of this renderer's last host frame (0 = rendered as one piece); out_ms (may be null,
 * room for 16) receives the device-timeline ms of every slice, out_stage_ms (may be null, room for
 * 16 x 8) every slice's stage times in the order of forma_renderer_stage_times. */
int forma_renderer_host_slices(const forma_renderer* r, double* out_ms, double* out_stage_ms) {
    if (!r || !r->r.last_slices || !r->slicer) return 0;
    const size_t n = std::min<size_t>(r->r.last_slices, 16);
    for (size_t i = 0; i < n && i < r->slicer->dev.size(); ++i) {
        if (out_ms) out_ms[i] = r->slicer->dev[i]->r.stage_ms[7];
        for (int k = 0; out_stage_ms && k < 8; ++k) out_stage_ms[8 * i + k] = r->slicer->dev[i]->r.stage_ms[k];
    }
    return (int)r->r.last_slices;
}

int forma_renderer_multi_device_count(const forma_renderer_multi* m) { return m ? (int)m->dev.size() : 0; }
int forma_renderer_multi_render(forma_renderer_multi* m, forma_composition* c, uint8_t* buffer, uint64_t width, uint64_t stride,
                                uint64_t height, const uint32_t channels[4], const float clear[4], const forma_rect* crop,
                                forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY,
                   [&] { return multi_render_impl(m, c, buffer, false, width, stride, height, channels, clear, crop, timings); });
}
int forma_renderer_multi_render_device(forma_renderer_multi* m, forma_composition* c, uint8_t* buffer_on_first_device,
                                       uint64_t width, uint64_t stride, uint64_t height, const uint32_t channels[4],
                                       const float clear[4], const forma_rect* crop, forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return multi_render_impl(m, c, buffer_on_first_device, true, width, stride, height, channels, clear, crop, timings);
    });
}
int forma_renderer_multi_render_format(forma_renderer_multi* m, forma_composition* c, void* buffer, uint32_t format, uint64_t width,
                                       uint64_t stride, uint64_t height, const uint32_t channels[4], const float clear[4],
                                       const forma_rect* crop, forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return multi_render_impl(m, c, static_cast<uint8_t*>(buffer), false, width, stride, height, channels, clear, crop, timings,
                                 format);
    });
}
int forma_renderer_multi_render_device_format(forma_renderer_multi* m, forma_composition* c, void* buffer_on_first_device,
                                              uint32_t format, uint64_t width, uint64_t stride, uint64_t height,
                                              const uint32_t channels[4], const float clear[4], const forma_rect* crop,
                                              forma_timings* timings) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] {
        return multi_render_impl(m, c, static_cast<uint8_t*>(buffer_on_first_device), true, width, stride, height, channels, clear,
                                 crop, timings, format);
    });
}
/* Tile-row boundaries of the bands the next frame will use (n + 1 values) and the
 * device-timeline ms every band took in the last frame (n values). */
int forma_renderer_multi_bands(const forma_renderer_multi* m, uint32_t* bounds, double* band_ms) {
    if (!m) return 0;
    for (size_t i = 0; bounds && i < m->bounds.size(); ++i) bounds[i] = m->bounds[i];
    for (size_t i = 0; band_ms && i < m->last_ms.size(); ++i) band_ms[i] = m->last_ms[i];
    return (int)m->dev.size();
}

static uint64_t row_costs_impl(forma_renderer* r, uint64_t cap, uint64_t* out) {
    Renderer& R = r->r;
    const uint32_t rows = R.last_tiles_y;
    if (!rows || !cap || !out) return rows;
    if (cudaSetDevice(R.device) != cudaSuccess) return 0;
    DeviceBuffer<unsigned long long> d;
    if (d.reserve(rows) != cudaSuccess) return 0;
    launch_row_costs(R.tile_range.ptr, R.last_tiles_x, rows, R.segs.ptr, R.last_segments, d.ptr, R.stream);
    std::vector<unsigned long long> h(rows);
    if (cudaMemcpyAsync(h.data(), d.ptr, rows * sizeof(unsigned long long), cudaMemcpyDeviceToHost, R.stream) != cudaSuccess ||
        cudaStreamSynchronize(R.stream) != cudaSuccess) {
        set_error("forma_renderer_row_costs: %s", cudaGetErrorString(cudaGetLastError()));
        return 0;
    }
    for (uint64_t i = 0; i < std::min<uint64_t>(cap, rows); ++i) out[i] = h[i];
    return rows;
}
uint64_t forma_renderer_row_costs(forma_renderer* r, uint64_t cap, uint64_t* out) {
    return guarded((uint64_t)0, [&] { return row_costs_impl(r, cap, out); });
}

int forma_set_option(const char* name, int value) {
    if (name)
        for (const OptionName& n : kOptionNames)
            if (!strcmp(n.name, name)) {
                if (value < n.lo || value > n.hi) break;
                options().*(n.field) = value;
                return FORMA_OK;
            }
    set_error("forma_set_option: unknown option or value out of range (%s = %d)", name ? name : "(null)", value);
    return FORMA_ERR_INVALID_ARGUMENT;
}
int forma_get_option(const char* name, int* value) {
    if (name && value)
        for (const OptionName& n : kOptionNames)
            if (!strcmp(n.name, name)) {
                *value = options().*(n.field);
                return FORMA_OK;
            }
    set_error("forma_get_option: unknown option %s", name ? name : "(null)");
    return FORMA_ERR_INVALID_ARGUMENT;
}

// Packed-fp32 self-test (see kernels_painter.cu): random and special operands (zeros,
// denormals, infinities, NaN, cancellation cases) through every packed helper of the painter.
static int selftest_impl(int device, uint64_t* mismatches) {
    if (!mismatches) return FORMA_ERR_INVALID_ARGUMENT;
    FORMA_CUDA_TRY(cudaSetDevice(device));
    const uint32_t n = 1u << 20;
    std::vector<float> h(3u * n);
    uint64_t sstate = 0x1234567ull;
    auto next = [&] {
        sstate += 0x9E3779B97F4A7C15ull;
        uint64_t z = sstate;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    };
    const uint32_t special[] = {0x00000000u, 0x80000000u, 0x00000001u, 0x007FFFFFu, 0x00800000u, 0x3F800000u, 0xBF800000u,
                                0x3F7FFFFFu, 0x3F800001u, 0x7F7FFFFFu, 0x7F800000u, 0xFF800000u, 0x7FC00000u, 0x33800000u};
    for (size_t i = 0; i < h.size(); ++i) {
        const uint64_t r = next();
        uint32_t bits;
        switch (r & 7u) {
            case 0: bits = special[(r >> 8) % (sizeof(special) / sizeof(special[0]))]; break;
            case 1: bits = (uint32_t)(r >> 32); break;                                  // any bit pattern
            case 2: bits = 0x3F800000u - (uint32_t)((r >> 32) & 0x3FFFFFu); break;      // just below 1
            default: {                                                                  // [0, 1) colours / coverages
                float f = (float)((r >> 40) & 0xFFFFFFu) / 16777216.0f;
                std::memcpy(&bits, &f, 4);
            }
        }
        std::memcpy(&h[i], &bits, 4);
    }
    DeviceBuffer<float> d;
    DeviceBuffer<uint32_t> out;
    FORMA_CUDA_TRY(d.reserve(h.size()));
    FORMA_CUDA_TRY(out.reserve(1));
    FORMA_CUDA_TRY(cudaMemcpy(d.ptr, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    FORMA_CUDA_TRY(cudaMemset(out.ptr, 0, sizeof(uint32_t)));
    launch_f32x2_selftest(d.ptr, d.ptr + n, d.ptr + 2u * n, n, out.ptr, 0);
    FORMA_CUDA_TRY(cudaGetLastError());
    uint32_t bad = 0;
    FORMA_CUDA_TRY(cudaMemcpy(&bad, out.ptr, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    *mismatches = bad;
    return FORMA_OK;
}
int forma_debug_selftest(int device, uint64_t* mismatches) {
    return guarded((int)FORMA_ERR_CAPACITY, [&] { return selftest_impl(device, mismatches); });
}

uint64_t forma_renderer_launch_count(const forma_renderer* r) { return r->r.launches; }
void forma_renderer_stage_times(const forma_renderer* r, double out_ms[8]) {
    const_cast<forma_renderer*>(r)->r.resolve_times();
    for (int i = 0; i < 8; ++i) out_ms[i] = r->r.stage_ms[i];
}
void forma_renderer_kernel_times(const forma_renderer* r, double out_ms[4], uint32_t out_launches[4]) {
    const_cast<forma_renderer*>(r)->r.resolve_times();
    for (int i = 0; i < 4; ++i) {
        out_ms[i] = r->r.kernel_ms[i];
        out_launches[i] = r->r.kernel_launches[i];
    }
}
void forma_renderer_counters(const forma_renderer* r, uint64_t out[8]) {
    out[6] = r->r.last_written_tiles;
    out[7] = r->r.last_tables_redone ? 2u : r->r.last_tables_sync_free ? 1u : 0u;
    out[0] = r->r.launches;
    out[1] = r->r.h2d_bytes;
    out[2] = r->r.d2h_bytes;
    out[3] = r->r.last_segments;
    out[4] = r->r.last_cells;
    out[5] = r->r.last_entries;
}
void forma_composition_evict(forma_composition* c) { c->c.evict(); }
uint64_t forma_composition_point_count(forma_composition* c) { return c->c.n_points; }
void forma_path_builder_extend(forma_path_builder* pb, const uint8_t* cmds, uint64_t n_cmds, const float* xy) {
    PathBuilder& b = pb->b;
    const float* p = xy;
    guarded_void([&] {
    for (uint64_t i = 0; i < n_cmds; ++i) {
        switch (cmds[i]) {
            case 0: b.move_to({p[0], p[1]}); p += 2; break;
            case 1: b.line_to({p[0], p[1]}); p += 2; break;
            case 2: b.quad_to({p[0], p[1]}, {p[2], p[3]}); p += 4; break;
            default: b.cubic_to({p[0], p[1]}, {p[2], p[3]}, {p[4], p[5]}); p += 6; break;
        }
    }
    });
}

static uint64_t renderer_lines_impl(forma_renderer* r, uint64_t cap, uint32_t* orders, float* x0, float* y0, float* dx,
                                    float* dy, float* a, float* b, float* c, float* d, uint32_t* lengths) {
    // Line records are never materialised by render(): line setup is fused into the
    // pixel-grid intersection kernel. For inspection they are produced here, by the same
    // device function (line_setup), from the arguments of the last render; the composition
    // of that render must still be alive.
    Renderer& R = r->r;
    if (!R.last_raster_valid || R.last_raster.n_points < 2) return 0;
    const uint32_t n = R.last_raster.n_points - 1u;
    if (!cap || !orders) return n;
    if (cudaSetDevice(R.device) != cudaSuccess) return 0;
    RasterArgs A = R.last_raster;
    A.band_lo = -3.0e38f;  // the reference's records know no tile bands
    A.band_hi = 3.0e38f;
    DeviceBuffer<uint32_t> d_orders, d_lengths;
    DeviceBuffer<float> d_f[8];
    if (d_orders.reserve(n) != cudaSuccess || d_lengths.reserve(n) != cudaSuccess) return 0;
    float* fp[8];
    for (int k = 0; k < 8; ++k) {
        if (d_f[k].reserve(n) != cudaSuccess) return 0;
        fp[k] = d_f[k].ptr;
    }
    launch_line_records(A, n, d_orders.ptr, fp, d_lengths.ptr, R.stream);
    const size_t m = (size_t)std::min<uint64_t>(cap, n);
    float* out[8] = {x0, y0, dx, dy, a, b, c, d};
    bool ok = cudaMemcpyAsync(orders, d_orders.ptr, m * 4, cudaMemcpyDeviceToHost, R.stream) == cudaSuccess &&
              cudaMemcpyAsync(lengths, d_lengths.ptr, m * 4, cudaMemcpyDeviceToHost, R.stream) == cudaSuccess;
    for (int k = 0; k < 8 && ok; ++k) ok = cudaMemcpyAsync(out[k], fp[k], m * 4, cudaMemcpyDeviceToHost, R.stream) == cudaSuccess;
    if (!ok || cudaStreamSynchronize(R.stream) != cudaSuccess) {
        set_error("forma_renderer_lines: %s", cudaGetErrorString(cudaGetLastError()));
        return 0;
    }
    uint32_t sum = 0;  // prefix_sum, segment.rs:90-98 (inclusive)
    for (size_t i = 0; i < m; ++i) {
        sum += lengths[i];
        lengths[i] = sum;
    }
    return n;
}
uint64_t forma_renderer_lines(forma_renderer* r, uint64_t cap, uint32_t* orders, float* x0, float* y0, float* dx, float* dy,
                              float* a, float* b, float* c, float* d, uint32_t* lengths) {
    return guarded((uint64_t)0, [&] { return renderer_lines_impl(r, cap, orders, x0, y0, dx, dy, a, b, c, d, lengths); });
}
uint64_t forma_renderer_segments(forma_renderer* r, uint64_t cap, uint64_t* out) {
    if (r->r.last_slices) {
        set_error("forma_renderer_segments: the last host frame was rendered in %u slices (option host_slices); "
                  "there is no single sorted segment array to inspect", r->r.last_slices);
        return 0;
    }
    uint64_t n = r->r.last_segments;
    if (out && cap && n) {
        cudaError_t e = cudaMemcpy(out, r->r.segs.ptr, std::min<uint64_t>(cap, n) * sizeof(uint64_t), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) {
            set_error("forma_renderer_segments: %s", cudaGetErrorString(e));
            return 0;
        }
    }
    return n;
}
static uint64_t rasterize_only_impl(forma_renderer* r, forma_composition* c, uint64_t width, uint64_t height,
                                    uint64_t cap, uint64_t* out) {
    Renderer& R = r->r;
    if (cudaSetDevice(R.device) != cudaSuccess) return 0;
    if (R.upload_tables(c->c, -1) || R.flush_geometry(c->c)) return 0;
    uint32_t n = 0;
    if (R.rasterize(c->c, (uint32_t)std::min<uint64_t>(width, 0xFFFFFFFFu), (uint32_t)std::min<uint64_t>(height, 0xFFFFFFFFu),
                    -3.0e38f, 3.0e38f, &n))
        return 0;
    if (cudaStreamSynchronize(R.stream) != cudaSuccess) return 0;
    if (out && cap && n &&
        cudaMemcpy(out, R.segs.ptr, std::min<uint64_t>(cap, n) * sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess)
        return 0;
    return n;
}
uint64_t forma_renderer_rasterize_only(forma_renderer* r, forma_composition* c, uint64_t width, uint64_t height,
                                       uint64_t cap, uint64_t* out) {
    return guarded((uint64_t)0, [&] { return rasterize_only_impl(r, c, width, height, cap, out); });
}
int forma_renderer_sort_u64(forma_renderer* r, uint64_t* keys, uint64_t n) {
    Renderer& R = r->r;
    if (n >= (1ull << 30)) {
        set_error("sort_u64: n too large");
        return FORMA_ERR_CAPACITY;
    }
    if (n < 2) return FORMA_OK;
    FORMA_CUDA_TRY(cudaSetDevice(R.device));
    FORMA_CUDA_TRY(R.segs.reserve(n + 1));  // one key of slack: the TMA downsweep copies an even number of keys
    FORMA_CUDA_TRY(R.segs_tmp.reserve(n + 1));
    FORMA_CUDA_TRY(R.sort_scratch.reserve(radix_scratch_bytes((uint32_t)n)));
    FORMA_CUDA_TRY(cudaMemcpyAsync(R.segs.ptr, keys, n * sizeof(uint64_t), cudaMemcpyHostToDevice, R.stream));
    // The caller's keys are on the host: take the field bounds from their OR.
    uint64_t all = 0;
    for (uint64_t i = 0; i < n; ++i) all |= keys[i];
    const uint64_t bound[3] = {(all >> 20) & 0x1FFFFFull, (all >> 41) & 0xFFFull, (all >> 53) & 0x7FFull};
    SortResult sr = launch_radix_sort(R.segs.ptr, R.segs_tmp.ptr, nullptr, nullptr, (uint32_t)n,
                                      make_sort_plan(segment_key_layout(), bound), R.sort_scratch.ptr, R.stream);
    R.launches += sr.launches;
    if (sr.in_tmp) Renderer::swap_buffers(R.segs, R.segs_tmp);
    FORMA_CUDA_TRY(cudaGetLastError());
    FORMA_CUDA_TRY(cudaMemcpyAsync(keys, R.segs.ptr, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, R.stream));
    FORMA_CUDA_TRY(cudaStreamSynchronize(R.stream));
    return FORMA_OK;
}

}  // extern "C"
