// Stage 4b: the painter — one warp per 16x16 tile. Replaces
// LayerWorkbench::drive_tile_painting + the optimiser passes
// (cpu/painter/layer_workbench/mod.rs:280-342, passes/*.rs),
// Painter::paint_layer / blend_at / clip_at / compute_srgb
// (cpu/painter/mod.rs:290-483) and LinearLayout::write
// (cpu/buffer/layout/mod.rs:265-282).
//
// Lane l owns eight horizontally consecutive pixels: row r = l / 2, columns 8 (l % 2) .. +8.
//   * the winding cover of a pixel is the carry-in of its row plus the covers of the
//     segments left of it in the same row: a running sum inside the lane and one shuffle
//     for the right half (the reference sweeps its columns left to right,
//     cpu/painter/mod.rs:388-404);
//   * the lane's eight cells are two 16-byte words of shared memory and its eight output
//     pixels one 32-byte run of the frame buffer;
//   * an entry without segments has one coverage value per lane.
// The reference's f32x8 is eight rows of one column; its "skip when all eight coverages
// are zero" (mod.rs:317-319) is reproduced from eight ballots where it can matter (any
// fill / blend other than a solid `Over`, for which blending with zero coverage is the
// identity on finite values).
//
// Per (tile, layer) entry the segments are scatter-added into packed cells — area in the
// high and cover in the low 16 bits of one word, one shared-memory atomic per segment —
// one entry ahead of the blend: while entry k is blended from one cell buffer, entry k + 1
// is accumulated into the other and the segments of entry k + 2 are in flight.
//
// Blend arithmetic runs on pixel pairs with Blackwell's packed fp32 instructions
// (fma.rn.f32x2 / mul.rn.f32x2 -> FFMA2 / FMUL2): each half is the IEEE operation the
// reference performs; additions and subtractions are written as fma(x, +-1, y), which is
// the same single rounding, so that no product is ever contracted into a sum.
//
// Warps are persistent and take tiles by ticket. Tiles with many entries come first
// (tile_index_kernel sorts them into four classes by entry count): a tile is painted by
// one warp from its first to its last layer, so the heaviest tile bounds the kernel's
// tail unless it starts early (longest-processing-time order).
//
// The output format is a template parameter of the kernel: RGBA8 encodes to sRGB bytes
// (compute_srgb), RGBA16F / RGBA32F store the same four linear values compute_srgb would
// receive, in channel order, as IEEE binary16 (round to nearest even) or binary32.
#include <cuda_fp16.h>
#include <mutex>
#include "paint_common.cuh"
#include "paint_math.cuh"

namespace forma {

struct PaintInputs {
    const uint64_t* segs;
    const EntryRec* recs;        // sorted entries (kernels_tables.cu: merge_entries_kernel)
    const uint2* tile_range;     // per tile: [begin, end) of its entries
    const uint32_t* heavy;       // kHeavyClasses lists of heavy tiles (linear ids), n_tiles_total each
    const uint32_t* heavy_count; // their lengths
    uint32_t n_tiles_total;
    uint8_t* eflags;             // per sorted entry: optimizer flags, initialised with EntryRec::flags0
    uint8_t* framebuffer;
    uint32_t* tile_counter;
    uint4* cache_solid_wide;     // FrameOut::cache_solid_wide (float formats)
};

__device__ __forceinline__ uint32_t meta_fill_rule(uint32_t m) { return m & 1u; }
__device__ __forceinline__ uint32_t meta_func(uint32_t m) { return (m >> 1) & 1u; }
__device__ __forceinline__ bool meta_is_clipped(uint32_t m) { return (m >> 2) & 1u; }
__device__ __forceinline__ uint32_t meta_fill_type(uint32_t m) { return (m >> 3) & 3u; }
__device__ __forceinline__ uint32_t meta_blend(uint32_t m) { return (m >> 5) & 15u; }

// ---------------------------------------------------------------------------
// Packed fp32 pairs
// ---------------------------------------------------------------------------
struct f2 {
    float x, y;
};
__device__ __forceinline__ unsigned long long f2_bits(f2 v) {
    return (unsigned long long)__float_as_uint(v.x) | ((unsigned long long)__float_as_uint(v.y) << 32);
}
__device__ __forceinline__ f2 f2_from(unsigned long long b) {
    return f2{__uint_as_float((uint32_t)b), __uint_as_float((uint32_t)(b >> 32))};
}
__device__ __forceinline__ f2 f2_splat(float v) { return f2{v, v}; }
#ifndef FORMA_SCALAR_PAIRS
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return f2_from(r);
}
__device__ __forceinline__ f2 mul2(f2 a, f2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return f2_from(r);
}
#else
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return f2{fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y)}; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { return f2{a.x * b.x, a.y * b.y}; }
#endif
// a + b and a - b as one fused operation each (exact product, one rounding: the IEEE sum).
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return fma2(a, f2_splat(1.0f), b); }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { return fma2(b, f2_splat(-1.0f), a); }
__device__ __forceinline__ f2 neg2(f2 a) { return f2{-a.x, -a.y}; }
__device__ __forceinline__ f2 min2(f2 a, f2 b) { return f2{fminf(a.x, b.x), fminf(a.y, b.y)}; }
__device__ __forceinline__ f2 max2(f2 a, f2 b) { return f2{fmaxf(a.x, b.x), fmaxf(a.y, b.y)}; }

// The 12 separable blend modes of the vector macro blend_function! (styling.rs:438-592) on a
// pixel pair, same operation order as vblend::blend (paint_math.cuh). `mode` is uniform.
__device__ __forceinline__ f2 hard2(f2 d, f2 s, f2 sel) {
    // sel <= 0.5 ? d * s * 2 : 2 * (d + s - fma(d, s, 0.5))
    const f2 lo = mul2(mul2(d, s), f2_splat(2.0f));
    const f2 hi = mul2(f2_splat(2.0f), sub2(add2(d, s), fma2(d, s, f2_splat(0.5f))));
    return f2{sel.x <= 0.5f ? lo.x : hi.x, sel.y <= 0.5f ? lo.y : hi.y};
}
__device__ __forceinline__ float soft1(float d, float s) {
    float dd = d <= 0.25f ? fmaf(fmaf(16.0f, d, -12.0f), d, 4.0f) * d : sqrtf(d);
    float k = fmaf(2.0f, s, -1.0f);
    return s <= 0.5f ? fmaf(d * (1.0f - d), k, d) : fmaf(dd - d, k, d);
}
__device__ __forceinline__ f2 blend_sep2(uint32_t mode, f2 d, f2 s) {
    switch (mode) {
        case 0: return s;
        case 1: return mul2(d, s);
        case 2: return add2(fma2(d, neg2(s), d), s);
        case 3: return hard2(d, s, d);
        case 4: return min2(d, s);
        case 5: return max2(d, s);
        case 6: return f2{s.x == 1.0f ? 1.0f : fminf(1.0f, d.x / (1.0f - s.x)), s.y == 1.0f ? 1.0f : fminf(1.0f, d.y / (1.0f - s.y))};
        case 7:
            return f2{s.x == 0.0f ? 0.0f : 1.0f - fminf(1.0f, (1.0f - d.x) / s.x),
                      s.y == 0.0f ? 0.0f : 1.0f - fminf(1.0f, (1.0f - d.y) / s.y)};
        case 8: return hard2(d, s, s);
        case 9: return f2{soft1(d.x, s.x), soft1(d.y, s.y)};
        case 10: {
            const f2 t = sub2(d, s);
            return f2{fabsf(t.x), fabsf(t.y)};
        }
        default: return add2(fma2(mul2(f2_splat(-2.0f), d), s, d), s);  // 11 Exclusion
    }
}

// blend_at's composition (cpu/painter/mod.rs:434-446) for a pixel pair and one channel:
//   current = fma(src, inv_dst_a * src_a, blended * (dst_a * src_a)); dst = fma(dst, 1 - src_a, current)
__device__ __forceinline__ f2 compose2(f2 dst, f2 src, f2 blended, f2 inv_dst_a_src_a, f2 dst_a_src_a, f2 inv_src_a) {
    const f2 cur = fma2(src, inv_dst_a_src_a, mul2(blended, dst_a_src_a));
    return fma2(dst, inv_src_a, cur);
}

// ---------------------------------------------------------------------------
// Out-of-line helpers for the rare paths (kept out of the kernel's instruction stream)
// ---------------------------------------------------------------------------
// One pixel of blend_at for any fill / blend mode.
__device__ __noinline__ float4 blend_pixel_generic(const StyleRec* __restrict__ st, const StopRec* __restrict__ stops,
                                                   const uint16_t* __restrict__ texels, float fx, float fy_base, int l,
                                                   float coverage, float clip, float4 dst) {
    float fill[4];
    if (st->fill_type == 0u) {
        fill[0] = st->color[0]; fill[1] = st->color[1]; fill[2] = st->color[2]; fill[3] = st->color[3];
    } else if (st->fill_type == 1u) {
        gradient_at(*st, stops, fx, fy_base, l, fill);
    } else {
        texture_at(*st, texels, fx, fy_base, l, fill);
    }
    float sa = fill[3] * coverage;
    if (clip >= 0.0f) sa *= clip;  // clip < 0: no mask applies
    float bl[3];
    vblend::blend(st->blend_mode, dst.x, dst.y, dst.z, fill[0], fill[1], fill[2], bl);
    float inv_dst_a = 1.0f - dst.w;
    float inv_dst_a_src_a = inv_dst_a * sa;
    float inv_src_a = 1.0f - sa;
    float dst_a_src_a = dst.w * sa;
    float cr = fmaf(fill[0], inv_dst_a_src_a, bl[0] * dst_a_src_a);
    float cg = fmaf(fill[1], inv_dst_a_src_a, bl[1] * dst_a_src_a);
    float cb = fmaf(fill[2], inv_dst_a_src_a, bl[2] * dst_a_src_a);
    return make_float4(fmaf(dst.x, inv_src_a, cr), fmaf(dst.y, inv_src_a, cg), fmaf(dst.z, inv_src_a, cb),
                       fmaf(dst.w, inv_src_a, sa));
}

__device__ __noinline__ uint32_t srgb_bytes_any_order(float r, float g, float b, float a, const uint32_t* ch) {
    return pixel_to_srgb_bytes(r, g, b, a, ch);
}

// The scalar blend of the solid-tile fold (all 16 modes) stays out of line too.
__device__ __noinline__ Rgba blend_solid(uint32_t mode, Rgba dst, Rgba src) { return sblend::blend(mode, dst, src); }

// sRGB encode of a pixel pair (compute_srgb, mod.rs:466-483), RGBA order.
__device__ __forceinline__ f2 srgb2(f2 l) {
    const f2 s = f2{sqrtf(l.x), sqrtf(l.y)};
    const f2 s3 = mul2(l, s);
    const f2 m = mul2(l, f2_splat(12.92f));
    const f2 n = fma2(f2_splat(0.20101772f), s3,
                      fma2(f2_splat(-0.51280147f), l, fma2(f2_splat(1.344401f), s, f2_splat(-0.030656587f))));
    return f2{l.x <= 0.0031308f ? m.x : n.x, l.y <= 0.0031308f ? m.y : n.y};
}
__device__ __forceinline__ void to_byte2(f2 v, uint32_t& b0, uint32_t& b1) {
    f2 sc = mul2(v, f2_splat(255.0f));
    sc.x = d_clamp(sc.x, 0.0f, 255.0f);
    sc.y = d_clamp(sc.y, 0.0f, 255.0f);
    const f2 val = add2(sc, f2_splat(__uint_as_float(0x4B000000u)));
    b0 = __float_as_uint(val.x) & 0xFFu;
    b1 = __float_as_uint(val.y) & 0xFFu;
}

__device__ __forceinline__ void store_tile_solid(const PaintScene& S, uint8_t* fb, uint32_t tx, uint32_t ty, uint32_t lane,
                                                 uint32_t rgba, bool vec_ok) {
    const uint32_t py = ty * 16u + (lane >> 1);
    const uint32_t px0 = tx * 16u + (lane & 1u) * 8u;
    if (py >= S.height || px0 >= S.width) return;
    uint8_t* row = fb + (size_t)py * S.stride + (size_t)px0 * 4u;
    if (vec_ok && px0 + 8u <= S.width) {
        const uint4 v = make_uint4(rgba, rgba, rgba, rgba);
        reinterpret_cast<uint4*>(row)[0] = v;
        reinterpret_cast<uint4*>(row)[1] = v;
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (px0 + (uint32_t)j < S.width) reinterpret_cast<uint32_t*>(row)[j] = rgba;
    }
}

// ---------------------------------------------------------------------------
// Float frames. A pixel is 16 B (RGBA32F: four f32) or 8 B (RGBA16F: four f16,
// __floats2half2_rn); its "wide" form is a uint4 holding those bytes (f16: in .x / .y).
// ---------------------------------------------------------------------------
__device__ __forceinline__ float4 select_channels(float r, float g, float b, float a, const uint32_t* ch) {
    const Rgba c{r, g, b, a};
    return make_float4(channel_of(c, ch[0]), channel_of(c, ch[1]), channel_of(c, ch[2]), channel_of(c, ch[3]));
}
__device__ __forceinline__ uint32_t half2_bits(float lo, float hi) {
    const __half2 h = __floats2half2_rn(lo, hi);  // .x (low 16 bits, first in memory) = lo
    return *reinterpret_cast<const uint32_t*>(&h);
}
template <uint32_t kFormat>
__device__ __forceinline__ uint4 wide_of(float4 v) {
    if (kFormat == kFormatRgba32f) return make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
    return make_uint4(half2_bits(v.x, v.y), half2_bits(v.z, v.w), 0u, 0u);
}
// One pixel at an address aligned to the element size only.
template <uint32_t kFormat>
__device__ __forceinline__ void store_pixel_scalar(uint8_t* p, uint4 w) {
    if (kFormat == kFormatRgba32f) {
        uint32_t* d = reinterpret_cast<uint32_t*>(p);
        d[0] = w.x; d[1] = w.y; d[2] = w.z; d[3] = w.w;
    } else {
        uint16_t* d = reinterpret_cast<uint16_t*>(p);
        d[0] = (uint16_t)w.x; d[1] = (uint16_t)(w.x >> 16); d[2] = (uint16_t)w.y; d[3] = (uint16_t)(w.y >> 16);
    }
}
// Pixels x, x + 1 of a lane's run (x even; p = their address). `vec`: the run is whole and
// 16-byte aligned: 16-byte stores (RGBA32F one per pixel, RGBA16F one per pair).
template <uint32_t kFormat>
__device__ __forceinline__ void store_pair(uint8_t* p, uint4 w0, uint4 w1, bool vec, uint32_t x, uint32_t width) {
    constexpr uint32_t kBpp = format_bytes_per_pixel(kFormat);
    if (vec) {
        if (kFormat == kFormatRgba32f) {
            reinterpret_cast<uint4*>(p)[0] = w0;
            reinterpret_cast<uint4*>(p)[1] = w1;
        } else {
            reinterpret_cast<uint4*>(p)[0] = make_uint4(w0.x, w0.y, w1.x, w1.y);
        }
    } else {
        if (x < width) store_pixel_scalar<kFormat>(p, w0);
        if (x + 1u < width) store_pixel_scalar<kFormat>(p + kBpp, w1);
    }
}

template <uint32_t kFormat>
__device__ __forceinline__ void store_tile_solid_wide(const PaintScene& S, uint8_t* fb, uint32_t tx, uint32_t ty, uint32_t lane,
                                                      uint4 w, bool vec_ok) {
    constexpr uint32_t kBpp = format_bytes_per_pixel(kFormat);
    const uint32_t py = ty * 16u + (lane >> 1);
    const uint32_t px0 = tx * 16u + (lane & 1u) * 8u;
    if (py >= S.height || px0 >= S.width) return;
    uint8_t* row = fb + (size_t)py * S.stride + (size_t)px0 * kBpp;
    const bool vec = vec_ok && px0 + 8u <= S.width;
#pragma unroll
    for (uint32_t j = 0; j < 8u; j += 2u) store_pair<kFormat>(row + j * kBpp, w, w, vec, px0 + j, S.width);
}

// Shared-memory word of pixel (local_x, local_y): row-major, ly * 16 + lx, i.e. the segment's
// (local_x, local_y) byte with its nibbles swapped. Lane l = 2 ly + lx / 8 owns the eight
// consecutive words l * 8 .. + 8 (two 16-byte accesses, two-way bank conflict: negligible
// next to the index arithmetic a swizzle would cost per segment).
__device__ __forceinline__ uint32_t cell_index_of(uint64_t s) {
    const uint32_t t = (uint32_t)(s >> 12);  // bits 7..4 local_x, 3..0 local_y
    return ((t & 15u) << 4) | ((t >> 4) & 15u);
}

// doubled_area_to_coverage (cpu/painter/mod.rs:76-94) by fill rule. The clamp of the
// non-zero rule only ever sees a non-negative, non-NaN value: min(v, 1) is the same result.
__device__ __forceinline__ float coverage_non_zero(int32_t doubled_area) {
    return fminf(fabsf((float)doubled_area * (1.0f / 512.0f)), 1.0f);
}
__device__ __forceinline__ float coverage_even_odd(int32_t doubled_area) {
    return (float)(512 - abs((doubled_area & 1023) - 512)) * (1.0f / 512.0f);
}

// Gradient::color_at (cpu/painter/styling.rs:58-144) for the pixel pair (x, x + 1) of one row,
// from the per-style record in shared memory (read as eight 16-byte words). Same operations
// in the same order as gradient_at (paint_math.cuh); d.recip() of every stop interval comes
// precomputed.
__device__ __forceinline__ void gradient_pair(const GradRec* gp, float x, float y_base, int lane_in_f32x8, f2& r, f2& gg, f2& b, f2& a) {
    const float4* gv = reinterpret_cast<const float4*>(gp);
    const float4 geo = gv[0];                                      // sx, sy, dx, dy
    const float4 hdr = gv[1];                                      // dot_recip, type, count, -
    const uint32_t type = __float_as_uint(hdr.y), count = __float_as_uint(hdr.z);
    const float4 st4 = gv[6], rc4 = gv[7];
    const float stop[4] = {st4.x, st4.y, st4.z, st4.w}, rcp_d[3] = {rc4.x, rc4.y, rc4.z};
    f2 t;
    const f2 xs = f2{x, x + 1.0f};
    if (type == 0u) {
        // tx = (x - sx) * dx * dot_recip; t = fma((lane + (y_base - sy)) * dy, dot_recip, tx)
        const f2 tx = mul2(mul2(sub2(xs, f2_splat(geo.x)), f2_splat(geo.z)), f2_splat(hdr.x));
        const float ty = y_base - geo.y;
        t = fma2(f2_splat(((float)lane_in_f32x8 + ty) * geo.w), f2_splat(hdr.x), tx);
    } else {
        const f2 px = sub2(xs, f2_splat(geo.x));
        const f2 px2 = mul2(px, px);
        const float py = (float)lane_in_f32x8 + (y_base - geo.y);
        const f2 q = mul2(fma2(f2_splat(py), f2_splat(py), px2), f2_splat(hdr.x));
        t = f2{sqrtf(q.x), sqrtf(q.y)};
    }
    float4 c_prev = gv[2];
    const float cp0[4] = {c_prev.x, c_prev.y, c_prev.z, c_prev.w};
    uint32_t bx[4], by[4];
    bool accx = t.x <= stop[0], accy = t.y <= stop[0];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        bx[k] = accx ? __float_as_uint(cp0[k]) : 0u;
        by[k] = accy ? __float_as_uint(cp0[k]) : 0u;
    }
    float start = 0.0f;
#pragma unroll
    for (uint32_t i = 1; i < 4u; ++i) {
        if (i < count) {
            const float4 c_cur = gv[2 + i];
            const bool mx = accx != (t.x < stop[i]), my = accy != (t.y < stop[i]);
            if (mx || my) {
                const f2 local_t = mul2(sub2(t, f2_splat(start)), f2_splat(rcp_d[i - 1]));
                const f2 neg_t = neg2(local_t);
                const float c0[4] = {c_prev.x, c_prev.y, c_prev.z, c_prev.w}, c1[4] = {c_cur.x, c_cur.y, c_cur.z, c_cur.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const f2 s0 = f2_splat(c0[k]);
                    const f2 v = fma2(local_t, f2_splat(c1[k]), fma2(neg_t, s0, s0));
                    if (mx) bx[k] |= __float_as_uint(v.x);
                    if (my) by[k] |= __float_as_uint(v.y);
                }
                accx = accx || mx;
                accy = accy || my;
            }
            start = stop[i];
            c_prev = c_cur;
        }
    }
    {
        const float4 c_last = gv[5];  // color[3] is the last stop (padding repeats it)
        const float cl[4] = {c_last.x, c_last.y, c_last.z, c_last.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (!accx) bx[k] |= __float_as_uint(cl[k]);
            if (!accy) by[k] |= __float_as_uint(cl[k]);
        }
    }
    r = f2{__uint_as_float(bx[0]), __uint_as_float(by[0])};
    gg = f2{__uint_as_float(bx[1]), __uint_as_float(by[1])};
    b = f2{__uint_as_float(bx[2]), __uint_as_float(by[2])};
    a = f2{__uint_as_float(bx[3]), __uint_as_float(by[3])};
}

// blend_at (cpu/painter/mod.rs:406-447) for one pixel pair of a layer with a separable blend mode
// and a solid or small-gradient fill. One out-of-line copy for the whole kernel: the twelve modes
// and the gradient, inlined per pair, do not fit the instruction cache. Arguments and result
// travel in registers.
//   ctl: blend mode | apply_clip << 8 | gradient fill << 9 | blend pixel x << 16 | blend pixel y << 17
struct PairPlanes {
    f2 r, g, b, a;
};
__device__ __noinline__ PairPlanes blend_pair_separable(PairPlanes d, f2 cov, f2 clip, uint32_t ctl, float x, float y_base,
                                                       int lane_in_f32x8, const GradRec* grad, float4 solid) {
    f2 fr = f2_splat(solid.x), fg = f2_splat(solid.y), fb = f2_splat(solid.z), fa = f2_splat(solid.w);
    if (ctl & 0x200u) gradient_pair(grad, x, y_base, lane_in_f32x8, fr, fg, fb, fa);
    f2 sa = mul2(fa, cov);
    if (ctl & 0x100u) sa = mul2(sa, clip);
    const uint32_t mode = ctl & 15u;
    const f2 br = blend_sep2(mode, d.r, fr), bg = blend_sep2(mode, d.g, fg), bb = blend_sep2(mode, d.b, fb);
    const f2 inv_dst_a = sub2(f2_splat(1.0f), d.a);
    const f2 inv_dst_a_src_a = mul2(inv_dst_a, sa);
    const f2 inv_src_a = sub2(f2_splat(1.0f), sa);
    const f2 dst_a_src_a = mul2(d.a, sa);
    const f2 nr = compose2(d.r, fr, br, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
    const f2 ng = compose2(d.g, fg, bg, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
    const f2 nb = compose2(d.b, fb, bb, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
    const f2 na = fma2(d.a, inv_src_a, sa);
    if (ctl & 0x10000u) {
        d.r.x = nr.x; d.g.x = ng.x; d.b.x = nb.x; d.a.x = na.x;
    }
    if (ctl & 0x20000u) {
        d.r.y = nr.y; d.g.y = ng.y; d.b.y = nb.y; d.a.y = na.y;
    }
    return d;
}

constexpr int kPaintWarpsPerBlock = 2;
constexpr uint32_t kPackedSegLimit = 2016u;  // segments per normalisation round of the packed cells (< 2048)

struct WarpSmem {
    uint32_t cells[2][256];  // packed (area << 16) + cover, double-buffered by entry parity
    float clip[256];         // clip mask, same layout
    EntryRec hdr[32];        // the 32 entry records of the current group (pad = current optimizer flags)
    GradRec grad;            // gradient of the entry being blended
};

// acc_segment (cpu/painter/mod.rs:257-271) for one segment: area and cover into the packed cell.
__device__ __forceinline__ void scatter_one(uint32_t* cells, uint64_t s) {
    const int32_t cv = (int32_t)(((uint32_t)s & 0x3Fu) ^ 0x20u) - 0x20;
    const int32_t dam = (int32_t)((uint32_t)(s >> 6) & 0x3Fu);
    atomicAdd(&cells[cell_index_of(s)], (uint32_t)((dam * cv) * 65536 + cv));
}

// Segments 64.. of a long entry (about one entry in ten has more than 64). Every
// kPackedSegLimit segments the low halves are folded back to i8 so that they cannot overflow
// 16 bits (areas wrap at i16, covers at i8, exactly like the reference's lanes).
__device__ __noinline__ void scatter_rest(const uint64_t* __restrict__ segs, uint32_t from, uint32_t s1, uint32_t* cells,
                                          uint32_t lane) {
    uint32_t done = 64u;
    for (uint32_t i0 = from; i0 < s1; i0 += 32u) {
        if (i0 + lane < s1) scatter_one(cells, segs[i0 + lane]);
        done += 32u;
        if (done >= kPackedSegLimit && i0 + 32u < s1) {
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t w = cells[k * 32 + lane];
                const int32_t lo = (int32_t)(int16_t)(w & 0xFFFFu);
                const uint32_t area = (w - (uint32_t)lo) & 0xFFFF0000u;
                cells[k * 32 + lane] = area + (uint32_t)(int32_t)(int8_t)lo;
            }
            __syncwarp();
            done = 0;
        }
    }
}

// Scatter-adds the segments [s0, s1) of one entry into `cells`. `pre0` / `pre1` hold the
// first two 32-segment chunks (requested one entry earlier).
__device__ __forceinline__ void scatter_entry(const uint64_t* __restrict__ segs, uint32_t s0, uint32_t s1, uint64_t pre0,
                                              uint64_t pre1, uint32_t* cells, uint32_t lane) {
    const uint32_t n = s1 - s0;
    if (lane < n) scatter_one(cells, pre0);
    if (lane + 32u < n) scatter_one(cells, pre1);
    if (n > 64u) scatter_rest(segs, s0 + 64u, s1, cells, lane);
}

template <int kMinBlocks, uint32_t kFormat>
__global__ void __launch_bounds__(kPaintWarpsPerBlock * 32, kMinBlocks) paint_kernel(PaintScene S, PaintInputs in, uint32_t n_tiles) {
    __shared__ __align__(16) WarpSmem s_warp[kPaintWarpsPerBlock];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    WarpSmem& W = s_warp[warp];
    const Rgba clear{S.clear[0], S.clear[1], S.clear[2], S.clear[3]};
    const bool rgba_order = S.channels[0] == 0u && S.channels[1] == 1u && S.channels[2] == 2u && S.channels[3] == 3u;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(in.framebuffer) | (uintptr_t)S.stride) & 15u) == 0u;
    const uint32_t ntx = S.tx_hi - S.tx_lo;
    const uint32_t row = lane >> 1, hx = lane & 1u;
    // The cells of this warp start (and are kept) zeroed.
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        W.cells[0][k * 32 + lane] = 0u;
        W.cells[1][k * 32 + lane] = 0u;
    }
    __syncwarp();

    // Ticket -> tile. Tickets [0, H) walk the heavy-tile lists (largest class first), the
    // remaining n_tiles tickets the tile rectangle in row-major order; a tile that is on a
    // list is skipped there. Lists hold tiles of the whole frame: those outside this
    // launch's rows / columns are skipped here.
    uint32_t hcount[kHeavyClasses], H = 0;
#pragma unroll
    for (int c = 0; c < kHeavyClasses; ++c) {
        hcount[c] = in.heavy ? in.heavy_count[c] : 0u;
        H += hcount[c];
    }
    const uint32_t n_tickets = H + n_tiles;
    auto resolve = [&](uint32_t ticket, uint32_t& tid, uint32_t& b, uint32_t& e) -> bool {
        if (ticket >= n_tickets) return false;
        if (ticket < H) {
            uint32_t t = ticket;
            int c = kHeavyClasses - 1;
#pragma unroll
            for (int q = kHeavyClasses - 1; q > 0; --q)
                if (c == q && t >= hcount[q]) {
                    t -= hcount[q];
                    c = q - 1;
                }
            tid = in.heavy[(size_t)c * in.n_tiles_total + t];
            const uint32_t ty = tid / S.tiles_x, tx = tid - ty * S.tiles_x;
            if (ty < S.ty_lo || ty >= S.ty_hi || tx < S.tx_lo || tx >= S.tx_hi) {
                tid = 0xFFFFFFFFu;  // not this launch's tile
                return true;
            }
            const uint2 r = in.tile_range[tid];
            b = r.x;
            e = r.y;
            return true;
        }
        const uint32_t lin = ticket - H;
        tid = (S.ty_lo + lin / ntx) * S.tiles_x + S.tx_lo + lin % ntx;
        const uint2 r = in.tile_range[tid];
        b = r.x;
        e = r.y;
        if (in.heavy && e - b >= kHeavyMin) tid = 0xFFFFFFFFu;  // painted from its list
        return true;
    };

    // Tickets are drawn two tiles ahead and the entry range of the next tile is loaded while
    // the current one is painted.
    uint32_t next_ticket = 0, cur_tid = 0, cur_b = 0, cur_e = 0;
    bool have = false;
    {
        uint32_t t0 = 0;
        if (lane == 0) t0 = atomicAdd(in.tile_counter, 1u);
        t0 = __shfl_sync(kFullMask, t0, 0);
        if (lane == 0) next_ticket = atomicAdd(in.tile_counter, 1u);
        have = resolve(t0, cur_tid, cur_b, cur_e);
    }
    while (have) {
        const uint32_t tid = cur_tid, b = cur_b, e = cur_e;
        {
            const uint32_t nxt = __shfl_sync(kFullMask, next_ticket, 0);
            have = resolve(nxt, cur_tid, cur_b, cur_e);
            if (lane == 0) next_ticket = atomicAdd(in.tile_counter, 1u);
        }
        if (tid == 0xFFFFFFFFu) continue;
        const uint32_t ty = tid / S.tiles_x, tx = tid - ty * S.tiles_x;

        // ---- optimizer passes (layer_workbench/passes/*.rs) ------------------
        // Pass A: per-entry facts, 32 entries at a time.
        // (has-segments / full / unchanged facts were computed when the entries were built.)
        bool any_clip = false, all_unchanged = true;
        for (uint32_t p0 = b; p0 < e; p0 += 32u) {
            uint32_t p = p0 + lane;
            uint32_t f = p < e ? (uint32_t)in.eflags[p] : kFlagUnchanged;
            any_clip |= __any_sync(kFullMask, (f & kFlagClipish) != 0u);
            all_unchanged = all_unchanged && !__any_sync(kFullMask, (f & kFlagUnchanged) == 0u);
        }

        // tile_unchanged pass (passes/tile_unchanged.rs:24-57) — only with a layer cache.
        const bool use_cache = S.cache_tiles != nullptr;
        uint32_t cache_x = 0, cache_solid = 0;
        bool layers_were_removed = true;  // PassesSharedState::reset
        if (use_cache) {
            uint2 c = S.cache_tiles[tid];
            const uint32_t layers = (e - b) & 0xFFFFFFu;
            const bool had = (c.x >> 31) != 0u;
            const uint32_t previous = c.x & 0xFFFFFFu;
            cache_solid = c.y;
            cache_x = (1u << 31) | (c.x & (1u << 30)) | layers;  // update_layer_count(Some(layers))
            bool is_unchanged = false;
            if (had) {
                layers_were_removed = layers < previous;
                is_unchanged = previous == layers && all_unchanged;
            }
            if (S.clear_unchanged && is_unchanged) {  // TileWriteOp::None
                if (lane == 0) S.cache_tiles[tid] = make_uint2(cache_x, cache_solid);
                continue;
            }
        }

        // Pass B: skip_trivial_clips (sequential; only tiles that contain clips).
        if (any_clip) {
            if (lane == 0) {
                bool has_clip = false, clip_full = false, clip_used = false;
                uint32_t clip_last = 0, clip_i = 0;
                for (uint32_t p = b; p < e; ++p) {
                    uint32_t f = in.eflags[p];
                    if (!(f & kFlagClipish)) {  // neither a clip nor a clipped layer
                        if (has_clip && in.recs[p].layer > clip_last) {
                            has_clip = false;
                            if (!clip_used) in.eflags[clip_i] |= (uint8_t)kFlagMaskedOut;
                        }
                        continue;
                    }
                    const uint32_t id = in.recs[p].layer;
                    if (!(f & kFlagClippedDraw)) {  // Func::Clip
                        clip_full = (f & kFlagFull) != 0;
                        clip_last = id + in.recs[p].clip_layers;
                        clip_i = p;
                        clip_used = false;
                        has_clip = true;
                        if (clip_full) f |= kFlagMaskedOut;
                    }
                    if (f & kFlagClippedDraw) {
                        if (has_clip && id <= clip_last) {
                            if (clip_full) f |= kFlagSkipClip;
                            else clip_used = true;
                        } else {
                            f |= kFlagMaskedOut;
                        }
                    }
                    in.eflags[p] = (uint8_t)f;
                    if (has_clip && id > clip_last) {
                        has_clip = false;
                        if (!clip_used) in.eflags[clip_i] |= (uint8_t)kFlagMaskedOut;
                    }
                }
                if (has_clip && !clip_used) in.eflags[clip_i] |= (uint8_t)kFlagMaskedOut;
            }
            __syncwarp();
        }

        // Pass C: skip_fully_covered_layers — the top-most full, unclipped, opaque
        // `Over` solid layer culls everything below it.
        uint32_t first_paint = b;  // MaskedVec::skip_until
        bool incomplete = false;   // an "interesting" incomplete cover at or above the opaque layer
        bool have_opaque = false;
        bool visible_unchanged = !layers_were_removed;  // skip_fully_covered_layers.rs:38-47
        for (uint32_t hi = e; hi > b && !have_opaque;) {
            uint32_t lo = hi - b >= 32u ? hi - 32u : b;
            uint32_t p = lo + lane;
            bool inc = false, cand = false, changed = false;
            if (p < hi) {
                uint32_t f = in.eflags[p];
                if (!(f & kFlagMaskedOut)) {
                    bool clipped = (f & kFlagClippedDraw) && !(f & kFlagSkipClip);
                    if (clipped || !(f & kFlagFull)) inc = true;
                    else if (f & kFlagOpaque) cand = true;
                    changed = !(f & kFlagUnchanged);
                }
            }
            uint32_t cand_mask = __ballot_sync(kFullMask, cand);
            uint32_t inc_mask = __ballot_sync(kFullMask, inc);
            uint32_t changed_mask = __ballot_sync(kFullMask, changed);
            if (cand_mask) {
                uint32_t top = 31u - (uint32_t)__clz((int)cand_mask);
                have_opaque = true;
                first_paint = lo + top;
                if (top < 31u && (inc_mask >> (top + 1u)) != 0u) incomplete = true;
                if ((changed_mask >> top) != 0u) visible_unchanged = false;  // layers visited before the break
            } else {
                if (inc_mask) incomplete = true;
                if (changed_mask) visible_unchanged = false;
            }
            hi = lo;
        }
        if (use_cache && have_opaque && !incomplete && visible_unchanged) {
            // Everything visible is unchanged: nothing to draw (skip_fully_covered_layers.rs:86-89).
            if (lane == 0) S.cache_tiles[tid] = make_uint2(cache_x, cache_solid);
            continue;
        }

        if (!incomplete) {
            // Every visible layer is full: fold with the scalar blend and emit a
            // solid tile (skip_fully_covered_layers.rs:81-118, mod.rs:686-704).
            Rgba dst = clear;
            uint32_t p = first_paint;
            if (have_opaque) {
                const EntryRec& r = in.recs[p];
                dst = Rgba{r.color[0], r.color[1], r.color[2], r.color[3]};
                ++p;
            }
            bool solid = true;
            for (; p < e; ++p) {
                if (in.eflags[p] & kFlagMaskedOut) continue;
                const EntryRec& r = in.recs[p];
                if (meta_func(r.meta) == 0u && meta_fill_type(r.meta) == 0u) {
                    dst = blend_solid(meta_blend(r.meta), dst, Rgba{r.color[0], r.color[1], r.color[2], r.color[3]});
                } else {
                    solid = false;
                    break;
                }
            }
            if (solid) {
                if constexpr (kFormat == kFormatRgba8) {
                    const uint32_t bytes = solid_to_srgb_bytes(dst, S.channels);
                    // CachedTile::convert_optimizer_op (cpu/painter/mod.rs:686-704): the same
                    // solid colour as last frame is not written again.
                    const bool same = use_cache && ((cache_x >> 30) & 1u) && cache_solid == bytes;
                    if (!same) store_tile_solid(S, in.framebuffer, tx, ty, lane, bytes, vec_ok);
                    if (lane == 0) {
                        if (use_cache) S.cache_tiles[tid] = make_uint2(cache_x | (1u << 30), bytes);
                        if (!same && S.written_list) S.written_list[atomicAdd(S.written_count, 1u)] = tid;
                    }
                } else {
                    // The same rule at the output precision: the colour is compared as the
                    // f16 / f32 bits the frame holds (side array in.cache_solid_wide).
                    const uint4 w = wide_of<kFormat>(select_channels(dst.r, dst.g, dst.b, dst.a, S.channels));
                    bool same = false;
                    if (use_cache && ((cache_x >> 30) & 1u)) {
                        const uint4 c = in.cache_solid_wide[tid];
                        same = c.x == w.x && c.y == w.y && c.z == w.z && c.w == w.w;
                    }
                    if (!same) store_tile_solid_wide<kFormat>(S, in.framebuffer, tx, ty, lane, w, vec_ok);
                    if (lane == 0) {
                        if (use_cache) {
                            S.cache_tiles[tid] = make_uint2(cache_x | (1u << 30), cache_solid);
                            in.cache_solid_wide[tid] = w;
                        }
                        if (!same && S.written_list) S.written_list[atomicAdd(S.written_count, 1u)] = tid;
                    }
                }
                continue;
            }
        }
        if (lane == 0) {
            // update_solid_color(None): the tile is painted
            if (use_cache) S.cache_tiles[tid] = make_uint2(cache_x & ~(1u << 30), cache_solid);
            if (S.written_list) S.written_list[atomicAdd(S.written_count, 1u)] = tid;
        }

        // ---- paint (layer_workbench/mod.rs:301-337, cpu/painter/mod.rs:290-347) ---
        // Pixel pair q = pixels 2 q, 2 q + 1 of the lane; (r, g, b, a) planes.
        f2 dr[4], dg[4], db[4], da[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            dr[q] = f2_splat(clear.r); dg[q] = f2_splat(clear.g); db[q] = f2_splat(clear.b); da[q] = f2_splat(clear.a);
        }
        bool clip_active = false;
        uint32_t clip_last = 0;
        const uint32_t x0 = tx * 16u + hx * 8u;            // first pixel column of the lane
        const float fy8 = (float)(ty * 16u + (row & 8u));  // y of lane 0 of the reference's f32x8 holding this row
        const int ly8 = (int)(row & 7u);                   // the row inside it
        const uint32_t grp_shift = (lane & 16u) + hx;      // ballot bits of this lane's f32x8 group: grp_shift + 2 i
        const uint4* hdr4 = reinterpret_cast<const uint4*>(W.hdr);

        for (uint32_t p0 = first_paint; p0 < e; p0 += 32u) {
            const uint32_t cnt = min(32u, e - p0);
            __syncwarp();  // the previous group's records are no longer read
            if (lane < cnt) {
                // Stage the record; its spare word carries the (possibly updated) optimizer flags,
                // and a masked-out entry gets an empty segment range: nothing to accumulate.
                const uint4* src = reinterpret_cast<const uint4*>(in.recs + p0 + lane);
                uint4* dstp = reinterpret_cast<uint4*>(&W.hdr[lane]);
                uint4 q0 = src[0];
                const uint4 q1 = src[1], q2 = src[2];
                uint4 q3 = src[3];
                q3.w = in.eflags[p0 + lane];
                if (q3.w & kFlagMaskedOut) q0.z = q0.y;
                dstp[0] = q0; dstp[1] = q1; dstp[2] = q2; dstp[3] = q3;
            }
            __syncwarp();

            // Pipeline prologue: entry 0 is accumulated now, the segments of entry 1 are requested.
            uint64_t nx0 = 0, nx1 = 0;  // first two chunks of the entry after the one being accumulated
            uint32_t grad_word = 0, grad_next = 0;
            {
                const uint4 h = hdr4[0];
                if (h.w & kMetaSmallGradient) grad_next = reinterpret_cast<const uint32_t*>(&S.grads[hdr4[3].x])[lane];
                const uint32_t s0 = h.y, s1 = h.z;
                uint64_t a0 = 0, a1 = 0;
                if (s0 + lane < s1) a0 = in.segs[s0 + lane];
                if (s0 + 32u + lane < s1) a1 = in.segs[s0 + 32u + lane];
                if (cnt > 1u) {
                    const uint4 g = hdr4[4];
                    if (g.y + lane < g.z) nx0 = in.segs[g.y + lane];
                    if (g.y + 32u + lane < g.z) nx1 = in.segs[g.y + 32u + lane];
                }
                if (s1 > s0) scatter_entry(in.segs, s0, s1, a0, a1, W.cells[0], lane);
                __syncwarp();
            }

            for (uint32_t k = 0; k < cnt; ++k) {
                // Request the segments of entry k + 2, accumulate entry k + 1 into the other buffer.
                {
                    const uint64_t c0 = nx0, c1 = nx1;
                    nx0 = nx1 = 0;
                    if (k + 2u < cnt) {
                        const uint4 g = hdr4[(k + 2u) * 4u];
                        if (g.y + lane < g.z) nx0 = in.segs[g.y + lane];
                        if (g.y + 32u + lane < g.z) nx1 = in.segs[g.y + 32u + lane];
                    }
                    grad_word = grad_next;  // word `lane` of this entry's gradient record (if it has one)
                    if (k + 1u < cnt) {
                        const uint4 g = hdr4[(k + 1u) * 4u];
                        if (g.w & kMetaSmallGradient)
                            grad_next = reinterpret_cast<const uint32_t*>(&S.grads[hdr4[(k + 1u) * 4u + 3u].x])[lane];
                        if (g.z > g.y) scatter_entry(in.segs, g.y, g.z, c0, c1, W.cells[(k + 1u) & 1u], lane);
                    }
                }
                const uint4 h0 = hdr4[k * 4u], h3 = hdr4[k * 4u + 3u];  // layer, seg0, seg1, meta | slot, clip_layers, flags0, flags
                const uint32_t flags = h3.w;
                if (flags & kFlagMaskedOut) {
                    __syncwarp();
                    continue;
                }
                const uint32_t meta = h0.w, layer = h0.x;
                const uint32_t fill_rule = meta_fill_rule(meta);

                // Running cover of this lane's row left of its first pixel (i8, wrapping like the
                // reference's lanes): the carry-in, plus the left half's covers for the right half.
                const uint32_t cw = reinterpret_cast<const uint32_t*>(&W.hdr[k].carry)[row >> 2];
                int32_t run = (int32_t)(int8_t)((cw >> (8u * (row & 3u))) & 0xFFu);
                f2 cov[4];  // coverage of the lane's pixel pairs
                if (h0.z > h0.y) {
                    // (the __syncwarp that ended the previous iteration made this buffer's atomics visible)
                    uint4* c4 = reinterpret_cast<uint4*>(W.cells[k & 1u]);
                    const uint4 w0 = c4[2u * lane], w1 = c4[2u * lane + 1u];
                    c4[2u * lane] = make_uint4(0u, 0u, 0u, 0u);
                    c4[2u * lane + 1u] = make_uint4(0u, 0u, 0u, 0u);
                    const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
                    int32_t area[8], cv[8], total = 0;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        cv[j] = (int32_t)(int16_t)(w[j] & 0xFFFFu);
                        area[j] = (int32_t)(w[j] + 0x8000u) >> 16;  // == (w - cover) >> 16: the high half as i16
                        total += cv[j];
                    }
                    const int32_t left = __shfl_xor_sync(kFullMask, total, 1);
                    if (hx) run += left;
                    // compute_doubled_areas, mod.rs:388-404: 32 * cover of the columns to the left + area
                    int32_t dbl[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        dbl[j] = 32 * (int32_t)(int8_t)run + area[j];
                        run += cv[j];
                    }
                    if (fill_rule == 0u) {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            cov[q] = f2{coverage_non_zero(dbl[2 * q]), coverage_non_zero(dbl[2 * q + 1])};
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            cov[q] = f2{coverage_even_odd(dbl[2 * q]), coverage_even_odd(dbl[2 * q + 1])};
                    }
                } else {
                    const float c = fill_rule == 0u ? coverage_non_zero(32 * run) : coverage_even_odd(32 * run);
#pragma unroll
                    for (int q = 0; q < 4; ++q) cov[q] = f2_splat(c);
                }

                if (clip_active && clip_last < layer) clip_active = false;  // mod.rs:302-306

                if (meta_func(meta) == 1u) {  // clip_at, mod.rs:449-464
                    if (!clip_active) {
                        clip_active = true;
                        clip_last = layer + h3.y;
                    }
                    float4* m4 = reinterpret_cast<float4*>(W.clip);
                    m4[2u * lane] = make_float4(cov[0].x, cov[0].y, cov[1].x, cov[1].y);
                    m4[2u * lane + 1u] = make_float4(cov[2].x, cov[2].y, cov[3].x, cov[3].y);
                    __syncwarp();
                    continue;
                }
                const bool apply_clip = meta_is_clipped(meta) && !(flags & kFlagSkipClip);
                bool nonzero = false;
#pragma unroll
                for (int q = 0; q < 4; ++q) nonzero = nonzero || cov[q].x != 0.0f || cov[q].y != 0.0f;
                if (!__any_sync(kFullMask, nonzero) || (apply_clip && !clip_active)) {  // mod.rs:317-323
                    __syncwarp();
                    continue;
                }
                f2 clip2[4];  // clip mask of the pairs; only read when apply_clip
                if (apply_clip) {
                    const float4* m4 = reinterpret_cast<const float4*>(W.clip);
                    const float4 m0 = m4[2u * lane], m1 = m4[2u * lane + 1u];
                    clip2[0] = f2{m0.x, m0.y}; clip2[1] = f2{m0.z, m0.w}; clip2[2] = f2{m1.x, m1.y}; clip2[3] = f2{m1.z, m1.w};
                } else {
                    clip2[0] = clip2[1] = clip2[2] = clip2[3] = f2_splat(0.0f);
                }

                const uint32_t mode = meta_blend(meta);
                const uint32_t fill_type = meta_fill_type(meta);
                const uint4 h2 = hdr4[k * 4u + 2u];  // the solid colour
                if (fill_type == 0u && mode == 0u) {
                    // blend_at (mod.rs:406-447) for a solid `Over` layer: blended == src, and zero
                    // coverage leaves the pixel as it is, so no f32x8 bookkeeping is needed.
                    const f2 cr = f2_splat(__uint_as_float(h2.x)), cg = f2_splat(__uint_as_float(h2.y));
                    const f2 cb = f2_splat(__uint_as_float(h2.z)), ca = f2_splat(__uint_as_float(h2.w));
                    if (apply_clip) {  // src_a = fill.a * coverage * mask (mod.rs:425-429)
#pragma unroll
                        for (int q = 0; q < 4; ++q) cov[q] = mul2(mul2(ca, cov[q]), clip2[q]);
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q) cov[q] = mul2(ca, cov[q]);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const f2 sa = cov[q];
                        const f2 inv_dst_a = sub2(f2_splat(1.0f), da[q]);
                        const f2 inv_dst_a_src_a = mul2(inv_dst_a, sa);
                        const f2 inv_src_a = sub2(f2_splat(1.0f), sa);
                        const f2 dst_a_src_a = mul2(da[q], sa);
                        dr[q] = compose2(dr[q], cr, cr, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
                        dg[q] = compose2(dg[q], cg, cg, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
                        db[q] = compose2(db[q], cb, cb, inv_dst_a_src_a, dst_a_src_a, inv_src_a);
                        da[q] = fma2(da[q], inv_src_a, sa);
                    }
                    __syncwarp();
                    continue;
                }

                // Everything else follows the reference's f32x8 rule exactly: a pixel is blended iff
                // some pixel of its f32x8 (same column, same half of the tile) has non-zero coverage.
                uint32_t active = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t b0 = __ballot_sync(kFullMask, cov[q].x != 0.0f), b1 = __ballot_sync(kFullMask, cov[q].y != 0.0f);
                    if ((b0 >> grp_shift) & 0x5555u) active |= 1u << (2 * q);
                    if ((b1 >> grp_shift) & 0x5555u) active |= 2u << (2 * q);
                }
                const int32_t slot = (int32_t)h3.x;
                const bool small_gradient = (meta & kMetaSmallGradient) != 0u;
                if (mode < 12u && (fill_type == 0u || small_gradient)) {
                    // Separable blend of a solid colour or a gradient of up to four stops: one
                    // out-of-line call per pixel pair that has a pixel to blend.
                    if (small_gradient) {
                        // The layer's gradient record (128 bytes, requested one entry ago) -> shared memory.
                        __syncwarp();
                        reinterpret_cast<uint32_t*>(&W.grad)[lane] = grad_word;
                        __syncwarp();
                    }
                    const float4 solid = make_float4(__uint_as_float(h2.x), __uint_as_float(h2.y), __uint_as_float(h2.z), __uint_as_float(h2.w));
                    const uint32_t ctl = mode | (apply_clip ? 0x100u : 0u) | (small_gradient ? 0x200u : 0u);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const uint32_t act = (active >> (2 * q)) & 3u;
                        if (act) {
                            const PairPlanes d = blend_pair_separable(PairPlanes{dr[q], dg[q], db[q], da[q]}, cov[q], clip2[q], ctl | (act << 16),
                                                                      (float)(x0 + 2u * (uint32_t)q), fy8, ly8, &W.grad, solid);
                            dr[q] = d.r; dg[q] = d.g; db[q] = d.b; da[q] = d.a;
                        }
                    }
                } else {
                    // Textures, gradients with more than four stops, non-separable modes: one
                    // out-of-line call per blended pixel.
                    const StyleRec* st = &S.styles[slot];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float fx = (float)(x0 + 2u * (uint32_t)q);
                        if ((active >> (2 * q)) & 1u) {
                            const float4 d = blend_pixel_generic(st, S.stops, S.texels, fx, fy8, ly8, cov[q].x, apply_clip ? clip2[q].x : -1.0f,
                                                                 make_float4(dr[q].x, dg[q].x, db[q].x, da[q].x));
                            dr[q].x = d.x; dg[q].x = d.y; db[q].x = d.z; da[q].x = d.w;
                        }
                        if ((active >> (2 * q + 1)) & 1u) {
                            const float4 d = blend_pixel_generic(st, S.stops, S.texels, fx + 1.0f, fy8, ly8, cov[q].y,
                                                                 apply_clip ? clip2[q].y : -1.0f, make_float4(dr[q].y, dg[q].y, db[q].y, da[q].y));
                            dr[q].y = d.x; dg[q].y = d.y; db[q].y = d.z; da[q].y = d.w;
                        }
                    }
                }
                __syncwarp();
            }
        }

        // compute_srgb + LinearLayout::write (mod.rs:466-483, layout/mod.rs:265-282).
        const uint32_t py = ty * 16u + row;
        if constexpr (kFormat != kFormatRgba8) {
            // Float frames: the accumulator as is, channel-selected, no encode.
            if (py < S.height && x0 < S.width) {
                constexpr uint32_t kBpp = format_bytes_per_pixel(kFormat);
                uint8_t* rowp = in.framebuffer + (size_t)py * S.stride + (size_t)x0 * kBpp;
                const bool vec = vec_ok && x0 + 8u <= S.width;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float4 p0, p1;
                    if (rgba_order) {
                        p0 = make_float4(dr[q].x, dg[q].x, db[q].x, da[q].x);
                        p1 = make_float4(dr[q].y, dg[q].y, db[q].y, da[q].y);
                    } else {
                        p0 = select_channels(dr[q].x, dg[q].x, db[q].x, da[q].x, S.channels);
                        p1 = select_channels(dr[q].y, dg[q].y, db[q].y, da[q].y, S.channels);
                    }
                    store_pair<kFormat>(rowp + 2u * (uint32_t)q * kBpp, wide_of<kFormat>(p0), wide_of<kFormat>(p1), vec,
                                        x0 + 2u * (uint32_t)q, S.width);
                }
            }
        } else if (py < S.height && x0 < S.width) {
            uint32_t out[8];
            if (rgba_order) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint32_t r0, r1, g0, g1, b0, b1, a0, a1;
                    to_byte2(srgb2(dr[q]), r0, r1);
                    to_byte2(srgb2(dg[q]), g0, g1);
                    to_byte2(srgb2(db[q]), b0, b1);
                    to_byte2(da[q], a0, a1);
                    out[2 * q] = r0 | (g0 << 8) | (b0 << 16) | (a0 << 24);
                    out[2 * q + 1] = r1 | (g1 << 8) | (b1 << 16) | (a1 << 24);
                }
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    out[2 * q] = srgb_bytes_any_order(dr[q].x, dg[q].x, db[q].x, da[q].x, S.channels);
                    out[2 * q + 1] = srgb_bytes_any_order(dr[q].y, dg[q].y, db[q].y, da[q].y, S.channels);
                }
            }
            uint8_t* rowp = in.framebuffer + (size_t)py * S.stride + (size_t)x0 * 4u;
            if (vec_ok && x0 + 8u <= S.width) {
                reinterpret_cast<uint4*>(rowp)[0] = make_uint4(out[0], out[1], out[2], out[3]);
                reinterpret_cast<uint4*>(rowp)[1] = make_uint4(out[4], out[5], out[6], out[7]);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (x0 + (uint32_t)j < S.width) reinterpret_cast<uint32_t*>(rowp)[j] = out[j];
            }
        }
    }
}

// Packs the tiles named in `list` (written by paint_kernel) into records of 256 pixels,
// row-major 16x16 (1 KB for RGBA8), so that a damaged frame costs a device->host copy
// proportional to the damage. One warp per tile. A pixel is kPerPixel elements of type E,
// each read at its own address: a float frame's stride need only be a multiple of E.
template <typename E, int kPerPixel>
__global__ void __launch_bounds__(256) gather_tiles_kernel(const uint8_t* __restrict__ fb, uint32_t stride, uint32_t width,
                                                           uint32_t height, uint32_t tiles_x,
                                                           const uint32_t* __restrict__ list,
                                                           const uint32_t* __restrict__ count, E* __restrict__ out) {
    const uint32_t n = *count;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t i = blockIdx.x * 8u + (threadIdx.x >> 5); i < n; i += gridDim.x * 8u) {
        const uint32_t tid = list[i];
        const uint32_t x0 = (tid % tiles_x) * 16u, y0 = (tid / tiles_x) * 16u;
#pragma unroll
        for (int k = 0; k < 8 * kPerPixel; ++k) {
            const uint32_t p = (uint32_t)k * 32u + lane;  // element index in the tile record
            const uint32_t px = p / (uint32_t)kPerPixel, e = p % (uint32_t)kPerPixel;  // pixel index in the tile, row-major
            const uint32_t x = x0 + (px & 15u), y = y0 + (px >> 4);
            E v = 0;
            if (x < width && y < height)
                v = *reinterpret_cast<const E*>(fb + (size_t)y * stride + ((size_t)x * kPerPixel + e) * sizeof(E));
            out[(size_t)i * (256u * kPerPixel) + p] = v;
        }
    }
}

void launch_gather_tiles(const PaintScene& S, uint32_t format, const uint8_t* framebuffer, void* packed, cudaStream_t st) {
    const int grid = device_sm_count() * 4;
    if (format == kFormatRgba32f)
        gather_tiles_kernel<uint32_t, 4><<<grid, 256, 0, st>>>(framebuffer, S.stride, S.width, S.height, S.tiles_x, S.written_list,
                                                               S.written_count, static_cast<uint32_t*>(packed));
    else if (format == kFormatRgba16f)
        gather_tiles_kernel<uint16_t, 4><<<grid, 256, 0, st>>>(framebuffer, S.stride, S.width, S.height, S.tiles_x, S.written_list,
                                                               S.written_count, static_cast<uint16_t*>(packed));
    else
        gather_tiles_kernel<uint32_t, 1><<<grid, 256, 0, st>>>(framebuffer, S.stride, S.width, S.height, S.tiles_x, S.written_list,
                                                               S.written_count, static_cast<uint32_t*>(packed));
}

// One thread per style slot: the GradRec of a gradient of up to four stops, with the very
// operations Gradient::get_t / color_at perform per call (styling.rs:59-66,107-108).
__global__ void grad_setup_kernel(const StyleRec* __restrict__ styles, const StopRec* __restrict__ stops, uint32_t n,
                                  GradRec* __restrict__ grads) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const StyleRec st = styles[i];
    GradRec g;
    g.pad = 0u;
    if (st.fill_type != 1u || st.stop_count < 2u || st.stop_count > 4u) {
        g.sx = g.sy = g.dx = g.dy = g.dot_recip = 0.0f;
        g.type = 0u;
        g.count = 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            g.stop[k] = g.rcp_d[k] = 0.0f;
#pragma unroll
            for (int c = 0; c < 4; ++c) g.color[k][c] = 0.0f;
        }
        grads[i] = g;
        return;
    }
    g.sx = st.start[0];
    g.sy = st.start[1];
    g.dx = st.end[0] - st.start[0];
    g.dy = st.end[1] - st.start[1];
    const float dot = g.dx * g.dx + g.dy * g.dy;
    g.dot_recip = d_rcp(dot);
    g.type = st.gradient_type;
    g.count = st.stop_count;
    const StopRec* sp = stops + st.stop_first;
    float start_stop = 0.0f;
#pragma unroll
    for (uint32_t k = 0; k < 4u; ++k) {
        const StopRec s = sp[k < st.stop_count ? k : st.stop_count - 1u];
#pragma unroll
        for (int c = 0; c < 4; ++c) g.color[k][c] = s.color[c];
        g.stop[k] = s.stop;
        if (k >= 1u) {
            g.rcp_d[k - 1u] = d_rcp(s.stop - start_stop);
            start_stop = s.stop;
        }
    }
    g.rcp_d[3] = 0.0f;
    grads[i] = g;
}
void launch_grad_setup(const StyleRec* styles, const StopRec* stops, uint32_t n_styles, GradRec* grads, cudaStream_t st) {
    if (n_styles) grad_setup_kernel<<<(n_styles + 127) / 128, 128, 0, st>>>(styles, stops, n_styles, grads);
}

// Self-test of the packed fp32 arithmetic (forma_debug_selftest): every packed helper against
// the scalar IEEE operation it stands for, on `n` operand triples. Returns mismatches in out[0].
__global__ void f32x2_selftest_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ c,
                                      uint32_t n, uint32_t* __restrict__ out) {
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) * 2u;
    if (i + 1u >= n) return;
    const f2 x{a[i], a[i + 1]}, y{b[i], b[i + 1]}, z{c[i], c[i + 1]};
    uint32_t bad = 0;
    auto same = [](float p, float q) { return __float_as_uint(p) == __float_as_uint(q) || (p != p && q != q); };
    const f2 f = fma2(x, y, z), m = mul2(x, y), s = add2(x, y), d = sub2(x, y);
    const f2 ms = add2(mul2(x, y), z);  // a product followed by a sum must stay two roundings
    bad += !same(f.x, fmaf(x.x, y.x, z.x)) + !same(f.y, fmaf(x.y, y.y, z.y));
    bad += !same(m.x, x.x * y.x) + !same(m.y, x.y * y.y);
    bad += !same(s.x, x.x + y.x) + !same(s.y, x.y + y.y);
    bad += !same(d.x, x.x - y.x) + !same(d.y, x.y - y.y);
    bad += !same(ms.x, (x.x * y.x) + z.x) + !same(ms.y, (x.y * y.y) + z.y);
    if (bad) atomicAdd(out, bad);
}
void launch_f32x2_selftest(const float* a, const float* b, const float* c, uint32_t n, uint32_t* out, cudaStream_t st) {
    f32x2_selftest_kernel<<<(n / 2 + 255) / 256, 256, 0, st>>>(a, b, c, n, out);
}

void launch_paint(const PaintScene& S, const uint64_t* segs, const EntryRec* recs, const uint2* tile_range, const uint32_t* heavy,
                  const uint32_t* heavy_count, uint8_t* eflags, uint8_t* framebuffer, uint32_t* tile_counter, cudaStream_t st,
                  const FrameOut& out) {
    if (S.tx_hi <= S.tx_lo || S.ty_hi <= S.ty_lo) return;
    uint32_t n_tiles = (S.tx_hi - S.tx_lo) * (S.ty_hi - S.ty_lo);
    cudaMemsetAsync(tile_counter, 0, sizeof(uint32_t), st);
    PaintInputs in{segs, recs, tile_range, heavy, heavy_count, S.tiles_x * S.tiles_y, eflags, framebuffer, tile_counter, out.cache_solid_wide};
    // Persistent warps: enough CTAs to fill every SM at the kernel's occupancy (per device).
    // Option paint_wide = 1 selects the build with up to 168 registers (6 CTAs / SM) instead of 128 (8 CTAs / SM).
    // Every output format has its own instantiation, so the occupancy is kept per format as well.
    static int blocks_per_sm[3][2][kMaxDevices] = {};
    static std::mutex config_mu;  // several host threads may render on one device
    const int wide = options().paint_wide ? 1 : 0;
    const uint32_t fmt = out.format <= kFormatRgba32f ? out.format : kFormatRgba8;
    using Kernel = void (*)(PaintScene, PaintInputs, uint32_t);
    static const Kernel kernels[3][2] = {{paint_kernel<8, kFormatRgba8>, paint_kernel<6, kFormatRgba8>},
                                         {paint_kernel<8, kFormatRgba16f>, paint_kernel<6, kFormatRgba16f>},
                                         {paint_kernel<8, kFormatRgba32f>, paint_kernel<6, kFormatRgba32f>}};
    const Kernel kernel = kernels[fmt][wide];
    int per_sm = 0;
    {
        std::lock_guard<std::mutex> lk(config_mu);
        int& slot = blocks_per_sm[fmt][wide][current_device_index()];
        if (!slot) {
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&slot, kernel, kPaintWarpsPerBlock * 32, 0);
            if (slot < 1) slot = 1;
        }
        per_sm = slot;
    }
    const uint32_t want = (uint32_t)(per_sm * device_sm_count());
    const uint32_t need = (n_tiles + kPaintWarpsPerBlock - 1) / kPaintWarpsPerBlock;
    kernel<<<min(want, need), kPaintWarpsPerBlock * 32, 0, st>>>(S, in, n_tiles);
}

}  // namespace forma
