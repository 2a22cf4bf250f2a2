// FLOAT-FRAME ORACLE — TEST INFRASTRUCTURE ONLY.
//
// The CPU oracle (oracle/forma_oracle.cpp, compiled into this library as it is) plus the
// float output formats of include/forma_b200.h: RGBA16F / RGBA32F frames hold, per pixel, the
// four f32 values compute_srgb / to_srgb_bytes would receive (cpu/painter/mod.rs:466-483,692),
// in channel order, as IEEE binary16 (round to nearest even) or binary32. The painter, the
// optimiser passes and every RGBA8 path are the oracle's own; only the last step of a tile (the
// encode and the write) and the layer cache's solid-colour comparison, which works at the output
// precision, are restated here. The library exports every fo_ symbol of the oracle and adds
//   fo_renderer_render_format   forma_renderer_render_format for host buffers
//   fo_encode_srgb              sRGB bytes of a float frame (what the RGBA8 frame holds)
//   fo_f32_to_f16               the RGBA16F conversion
//
// Build: see oracle_float/Makefile (the oracle's flags: -O3 -ffp-contract=off, OpenMP).

// The RGBA8 render and the cache's free are wrapped below: a cache remembers the format of its
// last frame, and a frame of another format starts it over like a new size does.
#define fo_renderer_render fo_renderer_render_rgba8
#define fo_layer_cache_free fo_layer_cache_free_base
#include "../oracle/forma_oracle.cpp"
#undef fo_renderer_render
#undef fo_layer_cache_free

#include <array>
#include <mutex>
#include <unordered_map>

namespace fo {
namespace ff {

enum : uint32_t { kFormatRgba8 = 0, kFormatRgba16f = 1, kFormatRgba32f = 2 };
inline size_t bpp_of(uint32_t f) { return f == kFormatRgba32f ? 16 : (f == kFormatRgba16f ? 8 : 4); }
inline size_t element_of(uint32_t f) { return f == kFormatRgba32f ? 4 : (f == kFormatRgba16f ? 2 : 1); }

// IEEE binary16 bits of v, round to nearest even; overflow -> +-inf, NaN stays NaN.
inline uint16_t f16_bits(float v) {
    _Float16 h = (_Float16)v;
    uint16_t b;
    std::memcpy(&b, &h, 2);
    return b;
}

// One pixel of a float frame: 16 (RGBA32F) or 8 (RGBA16F) bytes.
inline void encode(const float v[4], uint32_t format, uint8_t* out) {
    if (format == kFormatRgba32f) {
        std::memcpy(out, v, 16);
    } else {
        for (int k = 0; k < 4; ++k) {
            uint16_t h = f16_bits(v[k]);
            std::memcpy(out + 2 * k, &h, 2);
        }
    }
}

// What a layer cache keeps beyond the oracle's LayerCache: its last frame's format and, per tile,
// the solid colour at the output precision (the CachedTile's has-solid bit says whether it is set).
struct CacheExtra {
    uint32_t format = kFormatRgba8;
    std::vector<std::array<uint8_t, 16>> solid;
};
std::mutex extras_mu;
std::unordered_map<const LayerCache*, CacheExtra> extras;

CacheExtra& extra_of(const LayerCache* c) {
    std::lock_guard<std::mutex> lk(extras_mu);
    return extras[c];
}

struct Target {
    uint8_t* buffer;
    size_t width, height, stride;
    uint32_t format;
};

// LinearLayout::write (cpu/buffer/layout/mod.rs:265-282) at the format's pixel size.
inline void write_tile(const Target& rt, size_t tile_x, size_t tile_y, const uint8_t* colors_col_major, const uint8_t* solid) {
    const size_t bpp = bpp_of(rt.format);
    size_t x0 = tile_x * kTile, y0 = tile_y * kTile;
    for (size_t y = 0; y < (size_t)kTile && y0 + y < rt.height; ++y) {
        uint8_t* row = rt.buffer + (y0 + y) * rt.stride;
        for (size_t x = 0; x < (size_t)kTile && x0 + x < rt.width; ++x) {
            const uint8_t* src = colors_col_major ? colors_col_major + (x * kTile + y) * bpp : solid;
            std::memcpy(row + (x0 + x) * bpp, src, bpp);
        }
    }
}

// compute_srgb without the encode: the painter's channel-selected values, column-major.
inline void compute_linear(const Painter& p, const Channel ch[4], uint32_t format, uint8_t* out) {
    const size_t bpp = bpp_of(format);
    for (int i = 0; i < kTile * kTile; ++i) {
        float v[4];
        for (int k = 0; k < 4; ++k) {
            switch (ch[k]) {
                case kRed: v[k] = p.red[i]; break;
                case kGreen: v[k] = p.green[i]; break;
                case kBlue: v[k] = p.blue[i]; break;
                case kAlpha: v[k] = p.alpha[i]; break;
                case kZero: v[k] = 0.0f; break;
                default: v[k] = 1.0f; break;
            }
        }
        encode(v, format, out + i * bpp);
    }
}

// Workbench::drive_tile_painting (oracle/painter.hpp) with the solid tile encoded in `format` and
// compared with the cached one at that precision.
WriteOp drive_tile(Workbench& wb, Painter& painter, const TileContext& ctx, uint32_t format, uint8_t* cached_solid,
                   uint8_t solid_out[16]) {
    using Flow = Workbench::Flow;
    wb.populate_layers(ctx);
    Flow flow = wb.tile_unchanged_pass(ctx);
    Color solid;
    if (flow == Flow::Continue) {
        wb.skip_trivial_clips_pass(ctx);
        flow = wb.skip_fully_covered_layers_pass(ctx, &solid);
    }
    bool brk = false;
    WriteOp op = WriteOp::ColorBuffer;
    if (flow == Flow::BreakSolid) {
        float sel[4];
        for (int k = 0; k < 4; ++k) sel[k] = color_channel(solid, ctx.channels[k]);
        const size_t bpp = bpp_of(format);
        uint8_t px[16];
        encode(sel, format, px);
        bool unchanged = false;
        if (ctx.cached_tile) {
            bool had = ctx.cached_tile->has_solid();
            unchanged = had && std::memcmp(cached_solid, px, bpp) == 0;
            ctx.cached_tile->tags |= 1;
            std::memcpy(cached_solid, px, bpp);
        }
        std::memcpy(solid_out, px, bpp);
        op = unchanged ? WriteOp::None : WriteOp::Solid;
        brk = true;
    } else if (flow == Flow::BreakNone) {
        op = WriteOp::None;
        brk = true;
    } else if (ctx.cached_tile) {
        ctx.cached_tile->tags &= 2;  // update_solid_color(None)
    }
    if (brk) {
        for (auto& e : wb.ids) {
            CoverCarry cc;
            if (wb.cover_carry(ctx, e.id, &cc)) wb.next_queue.push_back(cc);
        }
        wb.next_tile();
        return op;
    }
    painter.clear(ctx.clear_color);
    for (size_t k = 0; k < wb.ids.size(); ++k) {
        uint32_t id = wb.ids[k].id;
        bool mask = k >= wb.skipped && wb.ids[k].mask;
        if (mask) {
            painter.clear_cells();
            if (const Workbench::SegRange* r = wb.segments_of(id))
                for (size_t i = r->first; i <= r->last; ++i) painter.acc_segment(ctx.segs[i]);
            if (const Cover* c = wb.cover(id)) painter.acc_cover(*c);
            const Props& props = ctx.props->get(id);
            bool apply_clip = false;
            if (props.func == kDraw) apply_clip = props.is_clipped && !wb.ids[k].skip_clipping;
            Cover out = painter.paint_layer(ctx.tile_x, ctx.tile_y, id, props, apply_clip);
            if (!out.is_empty(props.fill_rule)) wb.next_queue.push_back({out, id});
        } else {
            CoverCarry cc;
            if (wb.cover_carry(ctx, id, &cc)) wb.next_queue.push_back(cc);
        }
    }
    wb.next_tile();
    return WriteOp::ColorBuffer;
}

// paint_tile_row (oracle/painter.hpp) writing `rt.format` pixels.
void paint_row(Painter& painter, Workbench& wb, std::vector<uint8_t>& linear, size_t tile_y, const uint64_t* segs, size_t n,
               const PropsSource& props, const Channel ch[4], const Color& clear_color, bool has_prev_clear,
               const Color& prev_clear, CachedTile* cached_tiles, std::array<uint8_t, 16>* cached_solid, const Target& rt,
               const Rect* crop) {
    std::map<uint32_t, Cover> left;
    int16_t tile_x_start = crop ? (int16_t)crop->hor0 : 0;
    size_t pos = 0;
    while (pos < n && seg_tile_x(segs[pos]) < tile_x_start) {
        Cover& c = left[seg_layer(segs[pos])];
        int y = seg_local_y(segs[pos]);
        c.c[y] = (int8_t)(c.c[y] + seg_cover(segs[pos]));
        ++pos;
    }
    std::vector<CoverCarry> carries;
    for (auto& kv : left) carries.push_back({kv.second, kv.first});
    wb.init(std::move(carries));
    wb.next_queue.clear();
    wb.ids.clear();
    wb.skipped = 0;
    wb.segment_ranges.clear();
    wb.layers_were_removed = true;

    size_t width_in_tiles = (rt.width + kTile - 1) / kTile;
    for (size_t tile_x = 0; tile_x < width_in_tiles; ++tile_x) {
        if (crop && !(tile_x >= crop->hor0 && tile_x < crop->hor1)) continue;
        size_t begin = pos;
        while (pos < n && seg_tile_x(segs[pos]) == (int16_t)tile_x) ++pos;
        TileContext ctx;
        ctx.tile_x = tile_x;
        ctx.tile_y = tile_y;
        ctx.segs = segs + begin;
        ctx.n_segs = pos - begin;
        ctx.props = &props;
        ctx.has_cached_clear = has_prev_clear;
        ctx.cached_clear = prev_clear;
        ctx.cached_tile = cached_tiles ? cached_tiles + tile_x : nullptr;
        ctx.channels = ch;
        ctx.clear_color = clear_color;
        painter.clip_active = false;
        uint8_t solid[16];
        WriteOp op = drive_tile(wb, painter, ctx, rt.format, cached_solid ? cached_solid[tile_x].data() : nullptr, solid);
        if (op == WriteOp::Solid) {
            write_tile(rt, tile_x, tile_y, nullptr, solid);
        } else if (op == WriteOp::ColorBuffer) {
            compute_linear(painter, ch, rt.format, linear.data());
            write_tile(rt, tile_x, tile_y, linear.data(), nullptr);
        }
    }
}

// fo::render (oracle/forma_oracle.cpp) for a float target.
void render(Renderer& r, Composition& comp, const Target& rt, const uint32_t channels_in[4], const Color& clear_color,
            const Rect* crop, LayerCache* cache) {
    Channel ch[4];
    for (int k = 0; k < 4; ++k) {
        ch[k] = (Channel)channels_in[k];
        if (clear_color.a == 1.0f && ch[k] == kAlpha) ch[k] = kOne;
    }
    size_t wt = (rt.width + kTile - 1) / kTile, ht = (rt.height + kTile - 1) / kTile;
    CacheExtra* extra = nullptr;
    if (cache) {
        extra = &extra_of(cache);
        cache->tiles.resize(wt * ht);
        if (!cache->has_size || cache->width != rt.width || cache->height != rt.height || extra->format != rt.format) {
            cache->has_size = true;
            cache->width = rt.width;
            cache->height = rt.height;
            cache->clear();
        }
        extra->format = rt.format;
        extra->solid.resize(wt * ht);
    }
    comp.compact_geom();

    double t0 = now_ms();
    comp.fill_cpu_view(rt.width, rt.height, r.lines);
    double t1 = now_ms();
    rasterize(r.lines, r.segments);
    double t2 = now_ms();
    sort_segments(r.segments);
    double t3 = now_ms();

    PropsSource props;
    props.index(comp.layers);
    props.has_cache = cache != nullptr;
    props.cache_id = cache ? cache->id : 0;

    const uint64_t* segs = r.segments.data();
    size_t n = r.segments.size();
    size_t first = std::partition_point(segs, segs + n, [](uint64_t s) { return seg_tile_y(s) < 0; }) - segs;
    std::vector<size_t> row_start(ht + 1);
    for (size_t j = 0; j <= ht; ++j) {
        row_start[j] = std::partition_point(segs + first, segs + n, [j](uint64_t s) { return (size_t)seg_tile_y(s) < j; }) - segs;
    }
    bool has_prev_clear = cache && cache->has_clear;
    Color prev_clear = cache ? cache->clear_color : Color();
#pragma omp parallel
    {
        Painter painter;
        Workbench wb;
        std::vector<uint8_t> linear(kTile * kTile * 16);
#pragma omp for schedule(dynamic, 1)
        for (size_t j = 0; j < ht; ++j) {
            if (crop && !(j >= crop->vert0 && j < crop->vert1)) continue;
            paint_row(painter, wb, linear, j, segs + row_start[j], row_start[j + 1] - row_start[j], props, ch, clear_color,
                      has_prev_clear, prev_clear, cache ? cache->tiles.data() + j * wt : nullptr,
                      extra ? extra->solid.data() + j * wt : nullptr, rt, crop);
        }
    }
    double t4 = now_ms();

    if (cache) {
        cache->has_clear = true;
        cache->clear_color = clear_color;
        for (auto& kv : comp.layers) {
            if (kv.second->is_enabled) kv.second->is_unchanged |= (1u << cache->id);
            else kv.second->is_unchanged &= ~(1u << cache->id);
        }
    }
    r.last.line_setup_ms = t1 - t0;
    r.last.rasterize_ms = t2 - t1;
    r.last.sort_ms = t3 - t2;
    r.last.paint_ms = t4 - t3;
    r.last.n_lines = r.lines.size();
    r.last.n_segments = r.segments.size();
}

}  // namespace ff
}  // namespace fo

extern "C" {

int fo_renderer_render(void* rv, void* cv, uint8_t* buffer, uint64_t width, uint64_t stride, uint64_t height,
                       const uint32_t channels[4], const float clear[4], const fo_rect* crop, void* cache,
                       fo_timings* timings) {
    if (cache && width * 4 <= stride) {
        fo::ff::CacheExtra& extra = fo::ff::extra_of((LayerCache*)cache);
        if (extra.format != fo::ff::kFormatRgba8) ((LayerCache*)cache)->clear();
        extra.format = fo::ff::kFormatRgba8;
    }
    return fo_renderer_render_rgba8(rv, cv, buffer, width, stride, height, channels, clear, crop, cache, timings);
}

void fo_layer_cache_free(void* rv, void* cv) {
    {
        std::lock_guard<std::mutex> lk(fo::ff::extras_mu);
        fo::ff::extras.erase((LayerCache*)cv);
    }
    fo_layer_cache_free_base(rv, cv);
}

// forma_renderer_render_format for host buffers (include/forma_b200.h).
int fo_renderer_render_format(void* rv, void* cv, void* buffer, uint32_t format, uint64_t width, uint64_t stride,
                              uint64_t height, const uint32_t channels[4], const float clear[4], const fo_rect* crop,
                              void* cache, fo_timings* timings) {
    using namespace fo::ff;
    if (format > kFormatRgba32f) return 1;
    if (width * bpp_of(format) > stride || stride % element_of(format) || (uintptr_t)buffer % element_of(format)) return 1;
    if (format == kFormatRgba8)
        return fo_renderer_render(rv, cv, (uint8_t*)buffer, width, stride, height, channels, clear, crop, cache, timings);
    Renderer* r = (Renderer*)rv;
    Target rt{(uint8_t*)buffer, (size_t)width, (size_t)height, (size_t)stride, format};
    Rect rect;
    if (crop) {
        rect.hor0 = crop->hor_start / kTile;
        rect.hor1 = (crop->hor_end + kTile - 1) / kTile;
        rect.vert0 = crop->vert_start / kTile;
        rect.vert1 = (crop->vert_end + kTile - 1) / kTile;
    }
    Color cc{clear[0], clear[1], clear[2], clear[3]};
    fo::ff::render(*r, *(Composition*)cv, rt, channels, cc, crop ? &rect : nullptr, (LayerCache*)cache);
    if (timings) {
        timings->line_setup_ms = r->last.line_setup_ms;
        timings->rasterize_ms = r->last.rasterize_ms;
        timings->sort_ms = r->last.sort_ms;
        timings->paint_ms = r->last.paint_ms;
        timings->n_lines = r->last.n_lines;
        timings->n_segments = r->last.n_segments;
    }
    return 0;
}

// sRGB bytes of a float frame's pixels (`channels` as rendered, Alpha already One where the clear
// colour is opaque): slots holding R, G or B get to_byte(linear_to_srgb(v)), the others
// to_byte(v) -- what the RGBA8 frame holds for the channel orders of cpu/channel.rs.
void fo_encode_srgb(const float* rgba, uint64_t n_px, const uint32_t channels[4], uint8_t* out) {
    for (uint64_t i = 0; i < n_px * 4; ++i) {
        const uint32_t c = channels[i % 4];
        out[i] = c <= kBlue ? to_byte(linear_to_srgb(rgba[i])) : to_byte(rgba[i]);
    }
}

// The RGBA16F conversion of float frames (round to nearest even), n values.
void fo_f32_to_f16(const float* in, uint64_t n, uint16_t* out) {
    for (uint64_t i = 0; i < n; ++i) out[i] = fo::ff::f16_bits(in[i]);
}

}  // extern "C"
