"""Float frames (RGBA16F / RGBA32F) on the device against the CPU oracle.

Two frames are equal when np.array_equal(a, b, equal_nan=True) holds and their bit patterns
differ only where both values are zero (the sign of a zero) or both are NaN. Any other bit
difference is a painter value that differs from the oracle's. RGBA32F pins the painter's f32
arithmetic, which an RGBA8 comparison cannot see below the 8-bit rounding."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import scenes
import synth
import workloads
from forma_b200.binding import BGR0, BGR1, BGRA, RGB0, RGB1, RGBA, Color, Fill, FormaError, Format, Func, Point, Props, Rect, Style
from oracle_float import float_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLEAR = Color(1.0, 1.0, 1.0, 0.0)
FLOATS = {"rgba16f": np.float16, "rgba32f": np.float32}
SENTINEL = -7.25


@pytest.fixture(scope="module")
def oracle_api():
    """The oracle with float frames (oracle_float/): RGBA8 frames are the oracle's own."""
    return float_oracle.load()


def assert_same(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    if a.dtype == np.uint8:
        bad = a != b
    else:
        u = np.uint16 if a.dtype == np.float16 else np.uint32
        bad = (a.view(u) != b.view(u)) & ~((a == 0) & (b == 0)) & ~(np.isnan(a) & np.isnan(b))
    if bad.any():
        idx = np.argwhere(bad)
        first = tuple(idx[0])
        raise AssertionError(f"{what}: {len(idx)} values differ, first at {first}: cuda {a[first]!r} oracle {b[first]!r}")
    assert np.array_equal(a, b, equal_nan=a.dtype != np.uint8)


def effective_channels(channels, clear):
    return tuple(5 if (c == 3 and clear.a == 1.0) else c for c in channels)


def padded_frame(api, renderer, comp, w, h, dtype, channels=RGBA, clear=CLEAR, crop=None, cache=None, pad=0):
    """(frame [h, w, 4], padding [h, pad]): rows of w * 4 + `pad` values that start as a sentinel."""
    row = w * 4 + pad
    buf = np.full(h * row, SENTINEL if dtype != np.uint8 else 0xA5, dtype)
    renderer.render(comp, buf, w, h, channels, clear, crop, cache, stride=row * buf.itemsize)
    rows = buf.reshape(h, row)
    return rows[:, :w * 4].reshape(h, w, 4), rows[:, w * 4:]


def host_frame(*args, **kw):
    return padded_frame(*args, **kw)[0]


def comp_of(api, build):
    comp = api.Composition()
    build(api, comp)
    return comp


def both(cuda_api, oracle_api, build, w, h, dtype, **kw):
    out = []
    for api in (cuda_api, oracle_api):
        comp = api.Composition()
        build(api, comp)
        out.append(host_frame(api, api.Renderer(0), comp, w, h, dtype, **kw))
    return out


@pytest.mark.parametrize("fmt", sorted(FLOATS))
def test_e2e_scenes_match_oracle(cuda_api, oracle_api, fmt):
    for name in sorted(scenes.E2E):
        a, b = both(cuda_api, oracle_api, scenes.E2E[name], 64, 64, FLOATS[fmt])
        assert_same(a, b, name)


@pytest.mark.parametrize("fmt", sorted(FLOATS))
@pytest.mark.parametrize("seed,w,h", [(7, 320, 200), (11, 97, 61), (23, 1280, 720)])
def test_random_mixed_matches_oracle(cuda_api, oracle_api, fmt, seed, w, h):
    a, b = both(cuda_api, oracle_api, lambda api, c: synth.random_mixed(api, c, 300, w, h, seed), w, h, FLOATS[fmt])
    assert_same(a, b, f"random_mixed seed {seed}")


@pytest.mark.parametrize("name", ["circle256", "paris4k", "paris4k_grad", "cubics100k", "circles8k", "circles8k_1m"])
def test_workloads_rgba32f_match_oracle_and_rgba16f_is_the_cast(cuda_api, oracle_api, cuda_renderer, name):
    comp, w, h = workloads.build_scene(cuda_api, name)
    f32 = host_frame(cuda_api, cuda_renderer, comp, w, h, np.float32)
    f16 = host_frame(cuda_api, cuda_renderer, comp, w, h, np.float16)
    ocomp, _, _ = workloads.build_scene(oracle_api, name)
    want = host_frame(oracle_api, oracle_api.Renderer(0), ocomp, w, h, np.float32)
    assert_same(f32, want, name)
    with np.errstate(over="ignore"):
        assert_same(f16, f32.astype(np.float16), f"{name}: RGBA16F vs cast RGBA32F")
    if name in ("paris4k", "paris4k_grad"):  # the float frame encodes to the RGBA8 frame
        b8 = host_frame(cuda_api, cuda_renderer, comp, w, h, np.uint8)
        assert_same(float_oracle.encode_srgb(f32, RGBA), b8, f"{name}: encoded RGBA32F vs RGBA8")


def test_spaceship_200_frames_rgba16f_with_layer_cache(cuda_api, oracle_api):
    sides = []
    for api in (cuda_api, oracle_api):
        comp, w, h = workloads.build_scene(api, "spaceship1080p")
        r = api.Renderer(0)
        sides.append((comp, r, r.create_buffer_layer_cache(), np.zeros(w * h * 4, np.float16)))
    written = []
    for frame in range(1, 201):
        for comp, r, cache, buf in sides:
            comp.animate(frame)
            r.render(comp, buf, w, h, RGBA, CLEAR, None, cache)
        assert_same(sides[0][3], sides[1][3], f"spaceship frame {frame}")
        written.append(sides[0][1].counters()["written_tiles"])
    assert written[0] == ((w + 15) // 16) * ((h + 15) // 16)
    assert max(written[1:]) < (written[0] * 3) // 4
    assert sides[0][1].counters()["d2h_bytes"] > 0


@pytest.mark.parametrize("fmt", ["rgba8"] + sorted(FLOATS))
def test_device_and_tensor_frames_equal_host_frames(cuda_api, cuda_renderer, fmt):
    import torch
    dtype = {"rgba8": np.uint8, **FLOATS}[fmt]
    tdtype = {np.uint8: torch.uint8, np.float16: torch.float16, np.float32: torch.float32}[dtype]
    f = Format.of_dtype(dtype)
    w, h = 1920, 1080
    comp = cuda_api.Composition()
    synth.random_mixed(cuda_api, comp, 400, w, h, 31)
    want = host_frame(cuda_api, cuda_renderer, comp, w, h, dtype)
    dev = torch.zeros((h, w, 4), dtype=tdtype, device="cuda:0")
    cuda_renderer.render_device(comp, dev.data_ptr(), w, h, RGBA, CLEAR, format=f)
    torch.cuda.synchronize()
    assert_same(dev.cpu().numpy(), want, "render_device")
    r = cuda_api.Renderer(0)
    out = torch.zeros((h, w, 4), dtype=tdtype, device="cuda:0")
    r.render_tensor(comp, out, RGBA, CLEAR)
    torch.cuda.synchronize()
    assert_same(out.cpu().numpy(), want, "render_tensor")
    # a padded row stride: the tensor is a view of wider rows; the padding stays as it was
    base = torch.full((h, w + 3, 4), 7, dtype=tdtype, device="cuda:0")
    r.render_tensor(comp, base[:, :w], RGBA, CLEAR)
    torch.cuda.synchronize()
    got = base.cpu().numpy()
    assert_same(got[:, :w], want, "render_tensor, padded rows")
    assert (got[:, w:] == 7).all()


@pytest.mark.parametrize("fmt", sorted(FLOATS))
@pytest.mark.parametrize("order", ["RGBA", "BGRA", "RGB0", "BGR0", "RGB1", "BGR1"])
def test_channel_orders_and_clear_alpha(cuda_api, oracle_api, fmt, order):
    channels = {"RGBA": RGBA, "BGRA": BGRA, "RGB0": RGB0, "BGR0": BGR0, "RGB1": RGB1, "BGR1": BGR1}[order]
    for clear in (CLEAR, Color(0.1, 0.2, 0.3, 1.0)):
        a, b = both(cuda_api, oracle_api, lambda api, c: synth.random_mixed(api, c, 150, 200, 120, 5), 200, 120, FLOATS[fmt],
                    channels=channels, clear=clear)
        assert_same(a, b, f"{order} clear.a={clear.a}")


@pytest.mark.parametrize("fmt", sorted(FLOATS))
def test_padded_strides_partial_tiles_and_crops(cuda_api, oracle_api, fmt):
    dtype = FLOATS[fmt]
    build = lambda api, c: synth.random_mixed(api, c, 300, 1920, 1080, 13)  # 1080 = 67.5 tile rows
    for pad in (1, 5, 8):  # values of padding per row; 1 and 5: rows that are not 16-byte aligned (scalar stores)
        (a, pa), (b, _) = [padded_frame(api, api.Renderer(0), comp_of(api, build), 1920, 1080, dtype, pad=pad)
                           for api in (cuda_api, oracle_api)]
        assert_same(a, b, f"1080p pad {pad}")
        assert (pa == dtype(SENTINEL)).all()
    for crop in (Rect((100, 900), (37, 700)), Rect((1900, 1920), (1070, 1080)), Rect((0, 1920), (512, 1080))):
        a, b = both(cuda_api, oracle_api, build, 1920, 1080, dtype, crop=crop, pad=1)
        assert_same(a, b, f"crop {crop}")
    # odd widths: partial tile columns
    a, b = both(cuda_api, oracle_api, lambda api, c: synth.random_mixed(api, c, 100, 333, 77, 17), 333, 77, dtype, pad=2)
    assert_same(a, b, "333x77")


# --- layer cache -------------------------------------------------------------------------------

def solid(c):
    return Props(func=Func.Draw(Style(fill=Fill.Solid(c))))


def pixel_path(api, x, y):
    return (api.PathBuilder().move_to(Point(x, y)).line_to(Point(x, y + 1)).line_to(Point(x + 1, y + 1))
            .line_to(Point(x + 1, y)).line_to(Point(x, y)).build())


def box(api, x0, y0, x1, y1):
    return api.PathBuilder().move_to(Point(x0, y0)).line_to(Point(x0, y1)).line_to(Point(x1, y1)).line_to(Point(x1, y0)).build()


def animated_scene(api, dtype, frames=6, w=200, h=120):
    """tests/cache_scenarios.py animated_scene in a float format: a persistent cache, one buffer
    that keeps the pixels the cache does not rewrite."""
    r = api.Renderer(0)
    comp = api.Composition()
    cache = r.create_buffer_layer_cache()
    synth.random_mixed(api, comp, 60, w, h, 123)
    buf = np.full(w * h * 4, 0.2, dtype)
    shots = []
    for i in range(frames):
        if i == 1:
            comp.get(5).set_transform([1.0, 0.0, 0.0, 1.0, 7.0, 3.0])
        if i == 2:
            comp.get(9).disable()
            comp.get(20).set_props(solid(Color(0.2, 0.4, 0.9, 1.0)))
        if i == 3:
            comp.get(9).enable()
            comp.remove(30)
        if i == 4:
            comp.get(12).clear()
            comp.get(12).insert(synth.circle_path(api, 100.0, 60.0, 25.0))
        r.render(comp, buf, w, h, RGBA, Color(0.9, 0.9, 0.9, 1.0), None, cache)
        shots.append(buf.copy())
    return shots


def render_changed_layers_only(api, dtype):
    """cache_scenarios.render_changed_layers_only (forma/src/composition/mod.rs:1038-1105) in a float format."""
    T = 16
    r = api.Renderer(0)
    comp = api.Composition()
    cache = r.create_buffer_layer_cache()
    comp.insert(0, comp.create_layer().insert(pixel_path(api, 0, 0)).insert(pixel_path(api, T, 0)).set_props(
        solid(Color(1, 0, 0, 1))))
    comp.insert(1, comp.create_layer().insert(pixel_path(api, T + 1, 0)).insert(pixel_path(api, 2 * T, 0))
                .set_props(solid(Color(0, 1, 0, 1))))
    shots = []
    for i in range(2):
        if i == 1:
            comp.get(1).set_props(solid(Color(1, 0, 0, 1)))
        buf = np.zeros(3 * T * T * 4, dtype)
        r.render(comp, buf, 3 * T, T, RGBA, Color(0, 0, 0, 1), None, cache)
        shots.append(buf.reshape(T, 3 * T, 4))
    assert (shots[1][0, 0] == 0).all()  # first tile untouched
    assert shots[1][0, T].tolist() == [1, 0, 0, 1] and shots[1][0, 2 * T].tolist() == [1, 0, 0, 1]
    return shots


@pytest.mark.parametrize("fmt", sorted(FLOATS))
@pytest.mark.parametrize("scenario", [animated_scene, render_changed_layers_only])
def test_layer_cache_scenarios_match_oracle(cuda_api, oracle_api, fmt, scenario):
    got, want = scenario(cuda_api, FLOATS[fmt]), scenario(oracle_api, FLOATS[fmt])
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        assert_same(a, b, f"{scenario.__name__} frame {i}")


def _solid_scene(api, color):
    comp = api.Composition()
    # past every edge of the 32x32 frame: its four tiles hold no segment and fold to one solid colour
    comp.insert(0, comp.create_layer().insert(box(api, -8.0, -8.0, 40.0, 40.0)).set_props(solid(color)))
    return comp


@pytest.mark.parametrize("fmt,delta,rewritten", [
    ("rgba8", "f32_ulp", False),     # invisible at 8 bits
    ("rgba32f", "f32_ulp", True),    # one f32 ulp reaches a float frame
    ("rgba16f", "f32_ulp", False),   # below half an f16 ulp: the same halves
    ("rgba16f", "f16_ulp", True),
])
def test_solid_tile_cache_compares_at_output_precision(cuda_api, oracle_api, fmt, delta, rewritten):
    dtype = {"rgba8": np.uint8, **FLOATS}[fmt]
    r0 = np.float32(0.5)
    r1 = np.nextafter(r0, np.float32(1)) if delta == "f32_ulp" else np.float32(0.5 + 2.0 ** -11)
    frames = {}
    for api in (cuda_api, oracle_api):
        r = api.Renderer(0)
        cache = r.create_buffer_layer_cache()
        comp = _solid_scene(api, Color(float(r0), 0.25, 0.75, 1.0))
        buf = np.zeros(32 * 32 * 4, dtype)
        r.render(comp, buf, 32, 32, RGBA, CLEAR, None, cache)
        comp.get(0).set_props(solid(Color(float(r1), 0.25, 0.75, 1.0)))
        buf[:] = 0
        r.render(comp, buf, 32, 32, RGBA, CLEAR, None, cache)
        frames[api is cuda_api] = buf.copy()
        if api is cuda_api:
            assert r.counters()["written_tiles"] == (4 if rewritten else 0)
    assert_same(frames[True], frames[False], f"{fmt} {delta}")
    if rewritten and dtype == np.float32:
        assert (frames[True].reshape(-1, 4)[:, 0] == r1).all()


def test_cache_reused_with_another_format_redraws_every_tile(cuda_api, cuda_renderer):
    comp = cuda_api.Composition()
    w, h = 200, 120
    synth.random_mixed(cuda_api, comp, 60, w, h, 123)
    cache = cuda_renderer.create_buffer_layer_cache()
    tiles = ((w + 15) // 16) * ((h + 15) // 16)
    # a new format redraws every tile; the same format again with nothing changed redraws none
    for dtype, want in ((np.uint8, tiles), (np.float32, tiles), (np.float32, 0), (np.float16, tiles), (np.float16, 0),
                        (np.uint8, tiles)):
        host_frame(cuda_api, cuda_renderer, comp, w, h, dtype, cache=cache)
        assert cuda_renderer.counters()["written_tiles"] == want, (np.dtype(dtype).name, want)


@pytest.mark.parametrize("fmt", sorted(FLOATS))
def test_paint_wide_gives_the_same_float_frames(cuda_api, fmt):
    comp, w, h = workloads.build_scene(cuda_api, "paris4k_grad")
    saved = cuda_api.get_option("paint_wide")
    try:
        frames = []
        for wide in (0, 1):
            cuda_api.set_option("paint_wide", wide)
            frames.append(host_frame(cuda_api, cuda_api.Renderer(0), comp, w, h, FLOATS[fmt]))
    finally:
        cuda_api.set_option("paint_wide", saved)
    assert_same(frames[1], frames[0], "paint_wide 1 vs 0")


def test_float_host_frames_are_not_sliced(cuda_api, oracle_api):
    comp, w, h = workloads.build_scene(cuda_api, "paris4k")
    names = ("host_slices", "slice_min_points")
    saved = {n: cuda_api.get_option(n) for n in names}
    try:
        cuda_api.set_option("slice_min_points", 0)
        cuda_api.set_option("host_slices", 4)
        r = cuda_api.Renderer(0)
        host_frame(cuda_api, r, comp, w, h, np.uint8)
        assert len(r.host_slices()) == 4  # RGBA8 host frames of this scene are sliced
        got = host_frame(cuda_api, r, comp, w, h, np.float32)
        assert r.host_slices() == []
        assert r.counters()["d2h_bytes"] > 0
    finally:
        for n, v in saved.items():
            cuda_api.set_option(n, v)
    ocomp, _, _ = workloads.build_scene(oracle_api, "paris4k")
    assert_same(got, host_frame(oracle_api, oracle_api.Renderer(0), ocomp, w, h, np.float32), "paris4k RGBA32F with host_slices 4")


def _device_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("n_dev", [2, 4, 8])
@pytest.mark.parametrize("fmt", sorted(FLOATS))
def test_multi_gpu_float_frames_equal_single_gpu(cuda_api, cuda_renderer, n_dev, fmt):
    if _device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    import torch
    dtype = FLOATS[fmt]
    comp, w, h = workloads.build_scene(cuda_api, "paris4k")
    want = host_frame(cuda_api, cuda_renderer, comp, w, h, dtype)
    m = cuda_api.MultiRenderer(list(range(n_dev)))
    buf = np.full(h * w * 4, SENTINEL, dtype)
    for _ in range(2):  # first frame: equal bands; second: re-balanced
        m.render(comp, buf, w, h, RGBA, CLEAR)
        assert_same(buf.reshape(h, w, 4), want, f"{n_dev} GPUs host frame")
    dev = torch.zeros((h, w, 4), dtype=torch.float16 if dtype == np.float16 else torch.float32, device="cuda:0")
    m.render_device(comp, dev.data_ptr(), w, h, RGBA, CLEAR, format=Format.of_dtype(dtype))
    for d in range(n_dev):
        torch.cuda.synchronize(d)
    assert_same(dev.cpu().numpy(), want, f"{n_dev} GPUs device frame")


# --- argument checks (host side, before any launch) ----------------------------------------------

def test_invalid_arguments_raise(cuda_api, cuda_renderer):
    import torch
    comp = cuda_api.Composition()
    synth.random_mixed(cuda_api, comp, 10, 64, 64, 1)
    r = cuda_renderer
    dev = torch.zeros(64 * 64 * 16 + 64, dtype=torch.uint8, device="cuda:0")
    p = dev.data_ptr()
    with pytest.raises(FormaError):
        r.render_device(comp, p, 64, 64, format=7)
    ch, cc = (C.c_uint32 * 4)(*RGBA), (C.c_float * 4)(1.0, 1.0, 1.0, 0.0)
    assert cuda_api.renderer_render_device_format(r._h, comp._h, C.c_void_p(p), 3, 64, 64 * 16, 64, ch, cc, None, None, None) == 1
    assert cuda_api.renderer_render_format(r._h, comp._h, C.c_void_p(p), 9, 64, 64 * 16, 64, ch, cc, None, None, None) == 1
    for fmt, stride in ((Format.RGBA32F, 64 * 16 - 4), (Format.RGBA32F, 64 * 16 + 2), (Format.RGBA16F, 64 * 8 - 2),
                        (Format.RGBA16F, 64 * 8 + 1)):
        with pytest.raises(FormaError):
            r.render_device(comp, p, 64, 64, stride=stride, format=fmt)
    with pytest.raises(FormaError):  # buffer address not a multiple of the element size
        r.render_device(comp, p + 2, 64, 64, format=Format.RGBA32F)
    with pytest.raises(FormaError):
        r.render_device(comp, p + 1, 64, 64, format=Format.RGBA16F)
    host = np.zeros(64 * 64 * 8, np.float32)
    with pytest.raises(FormaError):
        r.render(comp, host, 64, 64, stride=64 * 16 - 4)
    if _device_count() >= 1:
        m = cuda_api.MultiRenderer([0])
        with pytest.raises(FormaError):
            m.render(comp, host, 64, 64, stride=64 * 16 + 2)
    # the renderer still works afterwards
    out = torch.zeros((64, 64, 4), dtype=torch.float32, device="cuda:0")
    r.render_tensor(comp, out, RGBA, CLEAR)
    torch.cuda.synchronize()


def test_render_tensor_rejects_bad_tensors(cuda_api, cuda_renderer):
    import torch
    comp = cuda_api.Composition()
    bad = [torch.zeros((8, 8, 4), dtype=torch.float32),                      # host tensor
           torch.zeros((8, 8, 4), dtype=torch.int32, device="cuda:0"),       # dtype
           torch.zeros((8, 8, 3), dtype=torch.float32, device="cuda:0"),     # shape
           torch.zeros((8, 8), dtype=torch.float32, device="cuda:0"),
           torch.zeros((8, 4, 8), dtype=torch.float32, device="cuda:0").permute(0, 2, 1)]  # last dims not contiguous
    if _device_count() >= 2:
        bad.append(torch.zeros((8, 8, 4), dtype=torch.float32, device="cuda:1"))  # another device
    for t in bad:
        with pytest.raises(FormaError):
            cuda_renderer.render_tensor(comp, t)


@pytest.mark.parametrize("fmt", sorted(FLOATS))
def test_cli_writes_the_linear_frame(cuda_api, tmp_path, fmt):
    from forma_b200 import svg
    gold = np.load(os.path.join(ROOT, "tests", "golden", "paris30k_excerpt.npz"))
    doc = tmp_path / "paris30k_excerpt.svg"
    doc.write_bytes(gold["svg"].tobytes())
    out = tmp_path / "frame.npy"
    w, h, scale = 640, 360, 0.5
    subprocess.check_call([sys.executable, "-m", "forma_b200.render", str(doc), str(out), "--width", str(w), "--height", str(h),
                           "--scale", str(scale), "--format", fmt], cwd=ROOT)
    got = np.load(out)
    assert got.shape == (h, w, 4) and got.dtype == FLOATS[fmt]
    comp = cuda_api.Composition()
    svg.compose(cuda_api, comp, svg.parse_svg(str(doc)), scale=scale)
    want = host_frame(cuda_api, cuda_api.Renderer(0), comp, w, h, FLOATS[fmt], clear=Color(1.0, 1.0, 1.0, 1.0))
    assert_same(got, want, "CLI frame")
    assert not (got == SENTINEL).all(axis=-1).any()
