"""Float frames (RGBA16F / RGBA32F) of the CPU oracle: the linear values its RGBA8 frame
encodes, in the same channel order, layout, crop and padding.

The RGBA32F frame run through fo_encode_srgb (the sRGB encode of compute_srgb) must give the
RGBA8 frame byte for byte, and the RGBA16F frame must be the RGBA32F frame cast to float16."""
import numpy as np
import pytest

import scenes
import synth
from forma_b200.binding import BGR0, BGR1, BGRA, RGB0, RGB1, RGBA, Color, FormaError, Rect
from oracle_float import float_oracle

@pytest.fixture(scope="module")
def oracle_api():
    """The oracle with float frames (oracle_float/)."""
    return float_oracle.load()


CHANNEL_ORDERS = {"RGBA": RGBA, "BGRA": BGRA, "RGB0": RGB0, "BGR0": BGR0, "RGB1": RGB1, "BGR1": BGR1}
CLEAR = Color(1.0, 1.0, 1.0, 0.0)


def effective_channels(channels, clear):
    """Alpha reads as One when clear.a == 1 (cpu/renderer.rs:87-92)."""
    return tuple(5 if (c == 3 and clear.a == 1.0) else c for c in channels)


def frames(api, build, w, h, channels=RGBA, clear=CLEAR, crop=None, pad=0):
    """RGBA8, RGBA16F and RGBA32F frames of one scene, each from a fresh composition and renderer.
    With `pad` > 0 the rows carry `pad` extra values that start as a sentinel."""
    out = []
    for dtype, sentinel in ((np.uint8, 0xA5), (np.float16, np.float16(-7.25)), (np.float32, np.float32(-7.25))):
        comp = api.Composition()
        build(api, comp)
        row = (w + pad) * 4
        buf = np.full(h * row, sentinel, dtype)
        api.Renderer().render(comp, buf, w, h, channels, clear, crop, stride=row * buf.itemsize)
        out.append(buf.reshape(h, w + pad, 4))
    return out


def same_bits(a, b):
    """Bitwise equality that treats every NaN as equal to every NaN."""
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    u = np.uint16 if a.dtype == np.float16 else np.uint32
    nan = np.isnan(a) & np.isnan(b)
    return bool(np.all((a.view(u) == b.view(u)) | nan))


def crop_mask(w, h, crop):
    """Pixels a frame with `crop` writes: the crop rounded out to whole tiles (cpu/renderer.rs:43-52)."""
    inside = np.zeros((h, w), bool)
    if crop is None:
        inside[:] = True
    else:
        (x0, x1), (y0, y1) = crop.horizontal, crop.vertical
        inside[(y0 // 16) * 16:-(-y1 // 16) * 16, (x0 // 16) * 16:-(-x1 // 16) * 16] = True
    return inside


def check(api, build, w, h, channels=RGBA, clear=CLEAR, crop=None, pad=0):
    b8, f16, f32 = frames(api, build, w, h, channels, clear, crop, pad)
    inside = crop_mask(w, h, crop)
    enc = float_oracle.encode_srgb(f32[:, :w][inside], effective_channels(channels, clear))
    assert np.array_equal(enc, b8[:, :w][inside]), f"{int((enc != b8[:, :w][inside]).any(axis=-1).sum())} pixels differ from RGBA8"
    assert same_bits(f16[:, :w], f32[:, :w].astype(np.float16))
    if pad:
        assert (b8[:, w:] == 0xA5).all() and (f16[:, w:] == np.float16(-7.25)).all() and (f32[:, w:] == -7.25).all()
    return b8, f16, f32


@pytest.mark.parametrize("name", sorted(scenes.E2E))
def test_e2e_scenes(oracle_api, name):
    check(oracle_api, lambda a, c: scenes.E2E[name](a, c), 64, 64)


@pytest.mark.parametrize("seed,w,h", [(7, 320, 200), (11, 97, 61), (23, 640, 360)])
def test_random_mixed(oracle_api, seed, w, h):
    check(oracle_api, lambda a, c: synth.random_mixed(a, c, 150, w, h, seed), w, h)


@pytest.mark.parametrize("order", sorted(CHANNEL_ORDERS))
@pytest.mark.parametrize("clear", [CLEAR, Color(0.2, 0.3, 0.4, 1.0)], ids=["clear_a0", "clear_a1"])
def test_channel_orders(oracle_api, order, clear):
    check(oracle_api, lambda a, c: synth.random_mixed(a, c, 80, 130, 70, 5), 130, 70, CHANNEL_ORDERS[order], clear)


def test_crop_writes_only_the_cropped_tiles(oracle_api):
    w, h = 150, 90
    b8, f16, f32 = check(oracle_api, lambda a, c: synth.random_mixed(a, c, 80, w, h, 9), w, h,
                         crop=Rect((20, 100), (17, 60)))
    inside = crop_mask(w, h, Rect((20, 100), (17, 60)))
    assert inside.sum() == 48 * 96
    assert (f32[~inside] == -7.25).all() and (f16[~inside] == np.float16(-7.25)).all() and (b8[~inside] == 0xA5).all()
    assert not (f32[inside] == -7.25).all(axis=-1).any()


def test_padded_stride_leaves_the_padding(oracle_api):
    check(oracle_api, lambda a, c: synth.random_mixed(a, c, 80, 75, 40, 3), 75, 40, pad=3)


F16_EDGES = np.array([
    0.0, -0.0, 1.0, -1.0, 0.5, 1.0 / 3.0, 65504.0, -65504.0, 65519.996, 65520.0, -65520.0, 1e6, np.inf, -np.inf, np.nan,
    2.0 ** -14, 2.0 ** -24, 2.0 ** -25, 2.0 ** -25 * 1.0000001, 3 * 2.0 ** -26, 2.0 ** -26, 5.9604645e-08, 6.0975552e-05,
    6.1035156e-05 - 2.0 ** -25, 1e-10, -1e-10, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 2049.0, 2051.0, 1.4e-45,
], np.float32)


def test_f16_conversion_matches_numpy(oracle_api):
    rng = np.random.default_rng(0)
    rand = np.concatenate([rng.standard_normal(20000).astype(np.float32) * 10.0 ** rng.integers(-9, 6, 20000),
                           rng.integers(0, 2 ** 32, 20000, dtype=np.uint64).astype(np.uint32).view(np.float32)])
    for v in (F16_EDGES, rand):
        got = float_oracle.f32_to_f16(v)
        with np.errstate(over="ignore"):
            want = v.astype(np.float16)
        assert same_bits(got, want)


@pytest.mark.parametrize("dtype,bad_stride", [(np.float16, 8 * 10 - 2), (np.float16, 8 * 10 + 1), (np.float32, 16 * 10 - 4),
                                              (np.float32, 16 * 10 + 2)])
def test_rejects_bad_strides(oracle_api, dtype, bad_stride):
    comp = oracle_api.Composition()
    buf = np.zeros(4 * 10 * 4 * 4, dtype)
    with pytest.raises(FormaError):
        oracle_api.Renderer().render(comp, buf, 10, 4, RGBA, CLEAR, stride=bad_stride)


def test_rejects_unknown_format(oracle_api):
    import ctypes as C
    comp = oracle_api.Composition()
    buf = np.zeros(64, np.float32)
    ch = (C.c_uint32 * 4)(*RGBA)
    cc = (C.c_float * 4)(1.0, 1.0, 1.0, 0.0)
    r = oracle_api.Renderer()
    st = oracle_api.renderer_render_format(r._h, comp._h, buf.ctypes.data_as(C.c_void_p), 3, 2, 32, 2, ch, cc, None, None, None)
    assert st == 1


def test_cache_starts_over_when_the_format_changes(oracle_api):
    """A layer cache remembers its last frame's format: a frame in another format writes every
    tile, the same format again with nothing changed writes none (prefilled buffers show which)."""
    w, h = 96, 64
    comp = oracle_api.Composition()
    synth.random_mixed(oracle_api, comp, 60, w, h, 123)
    r = oracle_api.Renderer()
    cache = r.create_buffer_layer_cache()
    for dtype, sentinel, written in ((np.uint8, 0xA5, True), (np.float32, -7.25, True), (np.float32, -7.25, False),
                                     (np.float16, -7.25, True), (np.float16, -7.25, False), (np.uint8, 0xA5, True)):
        buf = np.full(w * h * 4, sentinel, dtype)
        r.render(comp, buf, w, h, RGBA, CLEAR, None, cache)
        untouched = (buf.reshape(h, w, 4) == dtype(sentinel)).all(axis=-1)
        assert (not untouched.any()) if written else untouched.all(), (np.dtype(dtype).name, written)
