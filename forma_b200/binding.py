"""ctypes binding over the C ABI of include/forma_b200.h.

This is the reference-side stub a maintainer would write (INTEGRATION.md shows
the Rust `extern "C"` equivalent). The classes mirror the names and argument
meaning of the reference's public API (forma/src/lib.rs:128-154): `Point`,
`PathBuilder`, `Path`, `Order`, `Color`, `GradientBuilder`, `Props`/`Style`/
`Fill`, `Composition`, `Layer`, `Renderer`, channel constants `RGBA`, `BGRA`…

`Api(lib, prefix)` is generic over the symbol prefix so that the test-only CPU
oracle (oracle/oracle.py, prefix ``fo_``) can be driven by the same
scene-building code as the product library (prefix ``forma_``); nothing in
this module knows about the oracle.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

# ---------------------------------------------------------------------------
# Plain data (forma/src/styling.rs, forma/src/math/point.rs)
# ---------------------------------------------------------------------------


@dataclass(frozen=True)
class Point:
    x: float
    y: float


@dataclass(frozen=True)
class Color:
    """Linear RGBA, forma/src/styling.rs:28-33 (default: opaque black, :52-61)."""

    r: float = 0.0
    g: float = 0.0
    b: float = 0.0
    a: float = 1.0


class FillRule:
    NonZero = 0
    EvenOdd = 1


class GradientType:
    Linear = 0
    Radial = 1


class BlendMode:
    Over, Multiply, Screen, Overlay, Darken, Lighten, ColorDodge, ColorBurn = range(8)
    HardLight, SoftLight, Difference, Exclusion, Hue, Saturation, Color, Luminosity = range(8, 16)
    NAMES = [
        "Over", "Multiply", "Screen", "Overlay", "Darken", "Lighten", "ColorDodge", "ColorBurn",
        "HardLight", "SoftLight", "Difference", "Exclusion", "Hue", "Saturation", "Color", "Luminosity",
    ]


class Channel:
    Red, Green, Blue, Alpha, Zero, One = range(6)


# forma/src/cpu/channel.rs:57-62
RGBA = (Channel.Red, Channel.Green, Channel.Blue, Channel.Alpha)
BGRA = (Channel.Blue, Channel.Green, Channel.Red, Channel.Alpha)
RGB0 = (Channel.Red, Channel.Green, Channel.Blue, Channel.Zero)
BGR0 = (Channel.Blue, Channel.Green, Channel.Red, Channel.Zero)
RGB1 = (Channel.Red, Channel.Green, Channel.Blue, Channel.One)
BGR1 = (Channel.Blue, Channel.Green, Channel.Red, Channel.One)

LAYER_LIMIT = (1 << 21) - 1


class Format:
    """Output format of a frame (FORMA_FORMAT_*): RGBA8 is sRGB bytes (cpu::Renderer);
    RGBA16F / RGBA32F hold the painter's linear colour as is (gpu::Renderer's Rgba16Float
    texture), 4 values per pixel."""

    RGBA8, RGBA16F, RGBA32F = range(3)
    BYTES_PER_PIXEL = {RGBA8: 4, RGBA16F: 8, RGBA32F: 16}
    DTYPES = {RGBA8: np.uint8, RGBA16F: np.float16, RGBA32F: np.float32}
    NAMES = {"rgba8": RGBA8, "rgba16f": RGBA16F, "rgba32f": RGBA32F}

    @staticmethod
    def of_dtype(dtype) -> int:
        """uint8 -> RGBA8, float16 -> RGBA16F, float32 -> RGBA32F."""
        dt = np.dtype(dtype)
        for f, d in Format.DTYPES.items():
            if dt == np.dtype(d):
                return f
        raise ValueError(f"no frame format stores {dt}: use uint8, float16 or float32")


class OrderError(ValueError):
    pass


class GeomPresTransformError(ValueError):
    pass


class FormaError(RuntimeError):
    pass


@dataclass
class Gradient:
    type: int
    start: Point
    end: Point
    stops: List[Tuple[Color, float]]


class GradientBuilder:
    """forma/src/styling.rs:84-139. Stops are resolved by the library."""

    def __init__(self, start: Point, end: Point):
        self._type = GradientType.Linear
        self._start, self._end = start, end
        self._stops: List[Tuple[Color, float]] = []

    def type(self, t: int) -> "GradientBuilder":
        self._type = t
        return self

    def color(self, color: Color) -> "GradientBuilder":
        self._stops.append((color, -1.0))
        return self

    def color_with_stop(self, color: Color, stop: float) -> "GradientBuilder":
        if not (0.0 <= stop <= 1.0):
            raise ValueError("gradient stops must be between 0.0 and 1.0")
        self._stops.append((color, stop))
        return self

    def build(self) -> Optional[Gradient]:
        if len(self._stops) < 2:
            return None
        return Gradient(self._type, self._start, self._end, list(self._stops))


@dataclass
class Texture:
    """Texture{transform, image} with the image given as linear RGBA floats
    (Image::from_linear_rgba, styling.rs:320-327). transform = (ux, uy, vx, vy, tx, ty)."""

    transform: Tuple[float, float, float, float, float, float]
    linear_rgba: np.ndarray  # (h, w, 4) float32


@dataclass
class Fill:
    solid: Optional[Color] = None
    gradient: Optional[Gradient] = None
    texture: Optional[Texture] = None

    @staticmethod
    def Solid(c: Color) -> "Fill":
        return Fill(solid=c)

    @staticmethod
    def Gradient(g: Gradient) -> "Fill":
        return Fill(gradient=g)

    @staticmethod
    def Texture(t: Texture) -> "Fill":
        return Fill(texture=t)


@dataclass
class Style:
    is_clipped: bool = False
    fill: Fill = field(default_factory=lambda: Fill.Solid(Color()))
    blend_mode: int = BlendMode.Over


@dataclass
class Func:
    draw: Optional[Style] = None
    clip: Optional[int] = None

    @staticmethod
    def Draw(style: Style) -> "Func":
        return Func(draw=style)

    @staticmethod
    def Clip(n: int) -> "Func":
        return Func(clip=n)


@dataclass
class Props:
    fill_rule: int = FillRule.NonZero
    func: Func = field(default_factory=lambda: Func.Draw(Style()))


# ---------------------------------------------------------------------------
# C structs
# ---------------------------------------------------------------------------


class _CColor(C.Structure):
    _fields_ = [("r", C.c_float), ("g", C.c_float), ("b", C.c_float), ("a", C.c_float)]


class _CStop(C.Structure):
    _fields_ = [("color", _CColor), ("stop", C.c_float)]


class _CProps(C.Structure):
    _fields_ = [
        ("fill_rule", C.c_uint32), ("func", C.c_uint32), ("clip_layers", C.c_uint32),
        ("is_clipped", C.c_uint32), ("blend_mode", C.c_uint32), ("fill_type", C.c_uint32),
        ("color", _CColor), ("gradient_type", C.c_uint32),
        ("start", C.c_float * 2), ("end", C.c_float * 2),
        ("n_stops", C.c_uint32), ("stops", C.POINTER(_CStop)),
        ("tex_transform", C.c_float * 6), ("tex_width", C.c_uint32), ("tex_height", C.c_uint32),
        ("tex_linear_rgba", C.POINTER(C.c_float)),
    ]


class _CRect(C.Structure):
    _fields_ = [("hor_start", C.c_uint64), ("hor_end", C.c_uint64), ("vert_start", C.c_uint64), ("vert_end", C.c_uint64)]


class _CTimings(C.Structure):
    _fields_ = [
        ("line_setup_ms", C.c_double), ("rasterize_ms", C.c_double), ("sort_ms", C.c_double),
        ("paint_ms", C.c_double), ("n_lines", C.c_uint64), ("n_segments", C.c_uint64),
    ]


@dataclass
class Timings:
    line_setup_ms: float
    rasterize_ms: float
    sort_ms: float
    paint_ms: float
    n_lines: int
    n_segments: int


@dataclass
class Rect:
    """cpu::Rect::new(horizontal, vertical), pixel ranges (cpu/renderer.rs:38-53)."""

    horizontal: Tuple[int, int]
    vertical: Tuple[int, int]


# Every symbol include/forma_b200.h declares (without prefix), with signature.
_f, _u8p, _u32p, _u64p, _fp = C.c_float, C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_float)
_vp = C.c_void_p
SIGNATURES = {
    "last_error": (C.c_char_p, []),
    "path_builder_new": (_vp, []),
    "path_builder_free": (None, [_vp]),
    "path_builder_move_to": (None, [_vp, _f, _f]),
    "path_builder_line_to": (None, [_vp, _f, _f]),
    "path_builder_quad_to": (None, [_vp, _f, _f, _f, _f]),
    "path_builder_cubic_to": (None, [_vp, _f, _f, _f, _f, _f, _f]),
    "path_builder_rat_quad_to": (None, [_vp, _f, _f, _f, _f, _f]),
    "path_builder_rat_cubic_to": (None, [_vp, _f, _f, _f, _f, _f, _f, _f, _f]),
    "path_builder_extend": (None, [_vp, _u8p, C.c_uint64, _fp]),
    "path_builder_build": (_vp, [_vp]),
    "path_transform": (_vp, [_vp, _fp]),
    "path_free": (None, [_vp]),
    "path_segments": (C.c_int, [_vp, C.POINTER(_fp), C.POINTER(_fp), C.POINTER(_u8p), _u64p]),
    "path_program_stats": (None, [_vp, _u64p]),
    "composition_new": (_vp, []),
    "composition_free": (None, [_vp]),
    "composition_create_layer": (_vp, [_vp]),
    "composition_insert": (_vp, [_vp, C.c_uint32, _vp, C.POINTER(C.c_int)]),
    "composition_remove": (_vp, [_vp, C.c_uint32]),
    "composition_get": (_vp, [_vp, C.c_uint32]),
    "composition_get_mut_or_insert_default": (_vp, [_vp, C.c_uint32, C.POINTER(C.c_int)]),
    "composition_len": (C.c_uint64, [_vp]),
    "layer_drop": (None, [_vp, _vp]),
    "layer_geom_id": (C.c_uint64, [_vp]),
    "layer_insert": (C.c_int, [_vp, _vp, _vp]),
    "layer_clear": (C.c_int, [_vp, _vp]),
    "layer_set_is_enabled": (C.c_int, [_vp, _vp, C.c_int]),
    "layer_is_enabled": (C.c_int, [_vp]),
    "layer_set_transform": (C.c_int, [_vp, _vp, _fp]),
    "layer_set_props": (C.c_int, [_vp, _vp, C.POINTER(_CProps)]),
    "renderer_new": (_vp, [C.c_int]),
    "renderer_free": (None, [_vp]),
    "layer_cache_new": (_vp, [_vp]),
    "layer_cache_free": (None, [_vp, _vp]),
    "layer_cache_clear": (None, [_vp]),
    "renderer_render": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), _vp, C.POINTER(_CTimings)]),
    "renderer_render_device": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), _vp, C.POINTER(_CTimings)]),
    "renderer_render_format": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), _vp, C.POINTER(_CTimings)]),
    "renderer_render_device_format": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), _vp, C.POINTER(_CTimings)]),
    "renderer_launch_count": (C.c_uint64, [_vp]),
    "renderer_stage_times": (None, [_vp, C.POINTER(C.c_double)]),
    "renderer_counters": (None, [_vp, _u64p]),
    "renderer_host_slices": (C.c_int, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "renderer_kernel_times": (None, [_vp, C.POINTER(C.c_double), _u32p]),
    "renderer_set_stream": (None, [_vp, _vp]),
    "shared_frame_create": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]),
    "shared_frame_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "shared_frame_close": (C.c_int, [C.c_int, _vp]),
    "shared_frame_free": (C.c_int, [C.c_int, _vp]),
    "composition_evict": (None, [_vp]),
    "composition_point_count": (C.c_uint64, [_vp]),
    "renderer_lines": (C.c_uint64, [_vp, C.c_uint64, _u32p, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _u32p]),
    "renderer_segments": (C.c_uint64, [_vp, C.c_uint64, _u64p]),
    "renderer_rasterize_only": (C.c_uint64, [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _u64p]),
    "renderer_sort_u64": (C.c_int, [_vp, _u64p, C.c_uint64]),
    "debug_selftest": (C.c_int, [C.c_int, _u64p]),
    "renderer_multi_new": (_vp, [C.POINTER(C.c_int), C.c_int]),
    "renderer_multi_free": (None, [_vp]),
    "renderer_multi_device_count": (C.c_int, [_vp]),
    "renderer_multi_render": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), C.POINTER(_CTimings)]),
    "renderer_multi_render_device": (C.c_int, [_vp, _vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), C.POINTER(_CTimings)]),
    "renderer_multi_render_format": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), C.POINTER(_CTimings)]),
    "renderer_multi_render_device_format": (C.c_int, [_vp, _vp, _vp, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, _u32p, _fp, C.POINTER(_CRect), C.POINTER(_CTimings)]),
    "renderer_multi_bands": (C.c_int, [_vp, _u32p, C.POINTER(C.c_double)]),
    "renderer_row_costs": (C.c_uint64, [_vp, C.c_uint64, _u64p]),
    "set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "get_option": (C.c_int, [C.c_char_p, C.POINTER(C.c_int)]),
}


# The float-frame entry points: a library that renders RGBA8 frames only may lack them (its
# Renderer.render / render_device then refuse float buffers with FormaError).
FORMAT_SYMBOLS = ("renderer_render_format", "renderer_render_device_format", "renderer_multi_render_format",
                  "renderer_multi_render_device_format")


class Api:
    """Typed access to one shared library exporting `<prefix><name>` symbols."""

    def __init__(self, lib: C.CDLL, prefix: str, optional: Sequence[str] = ()):
        self.lib, self.prefix = lib, prefix
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, prefix + name)
            except AttributeError:
                if name in optional or name in FORMAT_SYMBOLS:
                    continue
                raise
            fn.restype, fn.argtypes = res, args
            setattr(self, name + "_fn" if name in ("set_option", "get_option") else name, fn)

    def format_call(self, name: str, what: str):
        """The float-frame entry point `name`, or FormaError when this library has none."""
        fn = getattr(self, name, None)
        if fn is None:
            raise FormaError(f"{what}: this library renders RGBA8 frames only (no {self.prefix}{name})")
        return fn

    def check(self, status: int, what: str) -> None:
        if status == 0:
            return
        msg = self.last_error().decode() if hasattr(self, "last_error") else ""
        if status == 2:
            raise OrderError(f"{what}: exceeded layer limit ({LAYER_LIMIT})")
        raise FormaError(f"{what}: status {status} {msg}")

    def set_option(self, name: str, value: int) -> None:
        """Schedule switch of the library (see include/forma_b200.h: forma_set_option)."""
        self.check(self.__dict__["set_option_fn"](name.encode(), int(value)), f"set_option({name})")

    def get_option(self, name: str) -> int:
        v = C.c_int(0)
        self.check(self.__dict__["get_option_fn"](name.encode(), C.byref(v)), f"get_option({name})")
        return int(v.value)

    # Constructors bound to this library -----------------------------------
    def PathBuilder(self) -> "PathBuilder":
        return PathBuilder(self)

    def Composition(self) -> "Composition":
        return Composition(self)

    def Renderer(self, device: int = 0) -> "Renderer":
        return Renderer(self, device)

    def MultiRenderer(self, devices: Sequence[int]) -> "MultiRenderer":
        return MultiRenderer(self, devices)

    def SharedFrame(self, device: int, nbytes: int, handle: Optional[bytes] = None) -> "SharedFrame":
        return SharedFrame(self, device, nbytes, handle)


class SharedFrame:
    """A frame in one GPU's HBM that other processes paint into over NVLink
    (forma_shared_frame_*): the owner passes `handle` (64 bytes) to the other
    ranks, which construct theirs with it; `ptr` goes to Renderer.render_device.
    `__cuda_array_interface__` lets torch / cupy view the bytes without a copy."""

    def __init__(self, api: "Api", device: int, nbytes: int, handle: Optional[bytes] = None):
        self._api, self.device, self.nbytes, self.owner = api, device, nbytes, handle is None
        p = C.c_void_p()
        if self.owner:
            buf = C.create_string_buffer(64)
            api.check(api.shared_frame_create(device, nbytes, C.byref(p), buf), "shared_frame_create")
            self.handle = buf.raw
        else:
            self.handle = bytes(handle)
            api.check(api.shared_frame_open(device, self.handle, C.byref(p)), "shared_frame_open")
        self.ptr = int(p.value)

    @property
    def __cuda_array_interface__(self):
        return {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 2}

    def close(self):
        if self.ptr:
            (self._api.shared_frame_free if self.owner else self._api.shared_frame_close)(self.device, C.c_void_p(self.ptr))
            self.ptr = 0


def _np_f32(ptr, n):
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy() if n else np.zeros(0, np.float32)


class Path:
    """forma/src/path.rs:670-766."""

    def __init__(self, api: Api, handle):
        self._api, self._h = api, handle

    def transform(self, m: Sequence[float]) -> "Path":
        arr = (C.c_float * 9)(*[float(v) for v in m])
        return Path(self._api, self._api.path_transform(self._h, arr))

    def program_stats(self) -> dict:
        """Host-side facts of the flatten program (CUDA library only; needs no GPU)."""
        out = (C.c_uint64 * 6)()
        self._api.path_program_stats(self._h, out)
        return dict(zip(("points", "quads", "splines", "point_records", "rational", "contour_ends"), [int(v) for v in out]))

    def segments(self):
        """Flattened points: (x, y, start_new_contour) numpy arrays."""
        x, y, c, n = _fp(), _fp(), _u8p(), C.c_uint64()
        self._api.check(self._api.path_segments(self._h, C.byref(x), C.byref(y), C.byref(c), C.byref(n)), "path_segments")
        k = n.value
        if k == 0:
            return np.zeros(0, np.float32), np.zeros(0, np.float32), np.zeros(0, np.uint8)
        return _np_f32(x, k), _np_f32(y, k), np.ctypeslib.as_array(c, shape=(k,)).copy()

    def __del__(self):
        try:
            self._api.path_free(self._h)
        except Exception:
            pass


class PathBuilder:
    """forma/src/path.rs:776-925."""

    def __init__(self, api: Api):
        self._api = api
        self._h = api.path_builder_new()

    def move_to(self, p: Point) -> "PathBuilder":
        self._api.path_builder_move_to(self._h, p.x, p.y)
        return self

    def line_to(self, p: Point) -> "PathBuilder":
        self._api.path_builder_line_to(self._h, p.x, p.y)
        return self

    def quad_to(self, p1: Point, p2: Point) -> "PathBuilder":
        self._api.path_builder_quad_to(self._h, p1.x, p1.y, p2.x, p2.y)
        return self

    def cubic_to(self, p1: Point, p2: Point, p3: Point) -> "PathBuilder":
        self._api.path_builder_cubic_to(self._h, p1.x, p1.y, p2.x, p2.y, p3.x, p3.y)
        return self

    def rat_quad_to(self, p1: Point, p2: Point, weight: float) -> "PathBuilder":
        self._api.path_builder_rat_quad_to(self._h, p1.x, p1.y, p2.x, p2.y, weight)
        return self

    def rat_cubic_to(self, p1: Point, p2: Point, p3: Point, w1: float, w2: float) -> "PathBuilder":
        self._api.path_builder_rat_cubic_to(self._h, p1.x, p1.y, p2.x, p2.y, p3.x, p3.y, w1, w2)
        return self

    def extend(self, cmds: np.ndarray, xy: np.ndarray) -> "PathBuilder":
        """Bulk move/line/quad/cubic (codes 0..3) with their points (float32, flat)."""
        cmds = np.ascontiguousarray(cmds, np.uint8)
        xy = np.ascontiguousarray(xy, np.float32)
        self._api.path_builder_extend(self._h, cmds.ctypes.data_as(_u8p), cmds.size, xy.ctypes.data_as(_fp))
        return self

    def build(self) -> Path:
        return Path(self._api, self._api.path_builder_build(self._h))

    def __del__(self):
        try:
            self._api.path_builder_free(self._h)
        except Exception:
            pass


def _lower_props(props: Props):
    """Props -> (_CProps, keepalive list)."""
    cp = _CProps()
    keep = []
    cp.fill_rule = props.fill_rule
    if props.func.clip is not None:
        cp.func = 1
        cp.clip_layers = int(props.func.clip)
        return cp, keep
    style = props.func.draw
    cp.func = 0
    cp.is_clipped = 1 if style.is_clipped else 0
    cp.blend_mode = style.blend_mode
    fill = style.fill
    if fill.solid is not None:
        cp.fill_type = 0
        c = fill.solid
        cp.color = _CColor(c.r, c.g, c.b, c.a)
    elif fill.gradient is not None:
        g = fill.gradient
        cp.fill_type = 1
        cp.gradient_type = g.type
        cp.start[0], cp.start[1] = g.start.x, g.start.y
        cp.end[0], cp.end[1] = g.end.x, g.end.y
        stops = (_CStop * len(g.stops))()
        for i, (c, s) in enumerate(g.stops):
            stops[i].color = _CColor(c.r, c.g, c.b, c.a)
            stops[i].stop = s
        keep.append(stops)
        cp.n_stops = len(g.stops)
        cp.stops = C.cast(stops, C.POINTER(_CStop))
    else:
        t = fill.texture
        cp.fill_type = 2
        img = np.ascontiguousarray(t.linear_rgba, dtype=np.float32)
        keep.append(img)
        for i in range(6):
            cp.tex_transform[i] = t.transform[i]
        cp.tex_height, cp.tex_width = img.shape[0], img.shape[1]
        cp.tex_linear_rgba = img.ctypes.data_as(_fp)
    return cp, keep


class Layer:
    """forma/src/composition/layer.rs:61-353. The handle is owned by the
    Composition; `drop()` is Rust's `Drop for Layer`."""

    def __init__(self, comp: "Composition", handle):
        self._c, self._h = comp, handle

    def insert(self, path: Path) -> "Layer":
        a = self._c._api
        a.check(a.layer_insert(self._c._h, self._h, path._h), "Layer::insert")
        return self

    def clear(self) -> "Layer":
        a = self._c._api
        a.check(a.layer_clear(self._c._h, self._h), "Layer::clear")
        return self

    def geom_id(self) -> int:
        return int(self._c._api.layer_geom_id(self._h))

    def set_props(self, props: Props) -> "Layer":
        a = self._c._api
        cp, keep = _lower_props(props)
        a.check(a.layer_set_props(self._c._h, self._h, C.byref(cp)), "Layer::set_props")
        del keep
        return self

    def set_transform(self, t: Sequence[float]) -> "Layer":
        """t = [ux, vx, uy, vy, tx, ty] as GeomPresTransform::try_from([f32; 6])."""
        a = self._c._api
        arr = (C.c_float * 6)(*[float(v) for v in t])
        st = a.layer_set_transform(self._c._h, self._h, arr)
        if st == 1:
            raise GeomPresTransformError("exceeded scaling factor")
        a.check(st, "Layer::set_transform")
        return self

    def is_enabled(self) -> bool:
        return bool(self._c._api.layer_is_enabled(self._h))

    def set_is_enabled(self, enabled: bool) -> "Layer":
        a = self._c._api
        a.check(a.layer_set_is_enabled(self._c._h, self._h, 1 if enabled else 0), "Layer::set_is_enabled")
        return self

    def enable(self) -> "Layer":
        return self.set_is_enabled(True)

    def disable(self) -> "Layer":
        return self.set_is_enabled(False)

    def drop(self) -> None:
        self._c._api.layer_drop(self._c._h, self._h)
        self._h = None


class Composition:
    """forma/src/composition/mod.rs:53-343."""

    def __init__(self, api: Api):
        self._api = api
        self._h = api.composition_new()

    def create_layer(self) -> Layer:
        return Layer(self, self._api.composition_create_layer(self._h))

    def insert(self, order: int, layer: Layer) -> Optional[Layer]:
        st = C.c_int(0)
        old = self._api.composition_insert(self._h, order, layer._h, C.byref(st))
        self._api.check(st.value, "Order::new")
        return Layer(self, old) if old else None

    def remove(self, order: int) -> Optional[Layer]:
        h = self._api.composition_remove(self._h, order)
        return Layer(self, h) if h else None

    def get(self, order: int) -> Optional[Layer]:
        h = self._api.composition_get(self._h, order)
        return Layer(self, h) if h else None

    get_mut = get

    def get_mut_or_insert_default(self, order: int) -> Layer:
        st = C.c_int(0)
        h = self._api.composition_get_mut_or_insert_default(self._h, order, C.byref(st))
        self._api.check(st.value, "Order::new")
        return Layer(self, h)

    def evict(self) -> None:
        """Drop device residency (next render re-uploads from pinned host memory)."""
        self._api.composition_evict(self._h)

    def point_count(self) -> int:
        return int(self._api.composition_point_count(self._h))

    def __len__(self) -> int:
        return int(self._api.composition_len(self._h))

    def is_empty(self) -> bool:
        return len(self) == 0

    def __del__(self):
        try:
            self._api.composition_free(self._h)
        except Exception:
            pass


class LayerCache:
    def __init__(self, renderer: "Renderer", handle):
        self._r, self._h = renderer, handle

    def clear(self):
        self._r._api.layer_cache_clear(self._h)

    def __del__(self):
        try:
            self._r._api.layer_cache_free(self._r._h, self._h)
        except Exception:
            pass


class Renderer:
    """forma/src/cpu/renderer.rs:56-224 — `render` has the same arguments:
    (composition, buffer(width, stride, height), channels, clear_color, crop)."""

    def __init__(self, api: Api, device: int = 0):
        self._api, self.device = api, device
        self._h = api.renderer_new(device)
        if not self._h:
            msg = api.last_error().decode() if hasattr(api, "last_error") else ""
            raise FormaError(f"Renderer::new failed (no CPU fallback exists): {msg}")

    def create_buffer_layer_cache(self) -> Optional[LayerCache]:
        h = self._api.layer_cache_new(self._h)
        return LayerCache(self, h) if h else None

    def _common(self, channels, clear_color, crop):
        ch = (C.c_uint32 * 4)(*channels)
        cc = (C.c_float * 4)(clear_color.r, clear_color.g, clear_color.b, clear_color.a)
        rect = None
        if crop is not None:
            rect = _CRect(crop.horizontal[0], crop.horizontal[1], crop.vertical[0], crop.vertical[1])
        return ch, cc, rect

    def render(self, composition: Composition, buffer: np.ndarray, width: int, height: int,
               channels=RGBA, clear_color: Color = Color(1.0, 1.0, 1.0, 1.0), crop: Optional[Rect] = None,
               layer_cache: Optional[LayerCache] = None, stride: Optional[int] = None, timings: bool = True) -> Optional[Timings]:
        """`buffer`: writable contiguous host array of >= height*stride bytes. Its dtype picks the
        frame format (Format.of_dtype): uint8 -> RGBA8 (sRGB bytes), float16 -> RGBA16F,
        float32 -> RGBA32F (linear values), 4 values per pixel; `stride` is in bytes
        (default width * bytes per pixel).
        timings=False passes a null `forma_timings*`: the call then does not query its stage events
        (stage_times() still can, afterwards)."""
        fmt = Format.of_dtype(buffer.dtype)
        stride = width * Format.BYTES_PER_PIXEL[fmt] if stride is None else stride
        assert buffer.flags["C_CONTIGUOUS"] and buffer.nbytes >= height * stride
        ch, cc, rect = self._common(channels, clear_color, crop)
        t = _CTimings() if timings else None
        args = (width, stride, height, ch, cc, C.byref(rect) if rect is not None else None,
                layer_cache._h if layer_cache else None, C.byref(t) if t is not None else None)
        if fmt == Format.RGBA8:
            st = self._api.renderer_render(self._h, composition._h, buffer.ctypes.data_as(C.c_void_p), *args)
        else:
            st = self._api.format_call("renderer_render_format", "Renderer::render")(self._h, composition._h, buffer.ctypes.data_as(C.c_void_p), fmt, *args)
        self._api.check(st, "Renderer::render")
        return Timings(t.line_setup_ms, t.rasterize_ms, t.sort_ms, t.paint_ms, t.n_lines, t.n_segments) if t is not None else None

    def render_device(self, composition: Composition, device_ptr: int, width: int, height: int,
                      channels=RGBA, clear_color: Color = Color(1.0, 1.0, 1.0, 1.0), crop: Optional[Rect] = None,
                      layer_cache: Optional[LayerCache] = None, stride: Optional[int] = None,
                      timings: bool = True, format: int = Format.RGBA8) -> Optional[Timings]:
        """The frame stays in device memory at `device_ptr`, in `format` (a Format constant);
        `stride` in bytes, default width * bytes per pixel."""
        if format not in Format.BYTES_PER_PIXEL:
            raise FormaError(f"Renderer::render_device: unknown format {format}")
        stride = width * Format.BYTES_PER_PIXEL[format] if stride is None else stride
        ch, cc, rect = self._common(channels, clear_color, crop)
        t = _CTimings() if timings else None
        args = (width, stride, height, ch, cc, C.byref(rect) if rect is not None else None,
                layer_cache._h if layer_cache else None, C.byref(t) if t is not None else None)
        if format == Format.RGBA8:
            st = self._api.renderer_render_device(self._h, composition._h, C.c_void_p(device_ptr), *args)
        else:
            st = self._api.format_call("renderer_render_device_format", "Renderer::render_device")(self._h, composition._h, C.c_void_p(device_ptr), format, *args)
        self._api.check(st, "Renderer::render_device")
        return Timings(t.line_setup_ms, t.rasterize_ms, t.sort_ms, t.paint_ms, t.n_lines, t.n_segments) if t is not None else None

    def render_tensor(self, composition: Composition, out, channels=RGBA, clear_color: Color = Color(1.0, 1.0, 1.0, 1.0),
                      crop: Optional[Rect] = None, layer_cache: Optional[LayerCache] = None,
                      timings: bool = True) -> Optional[Timings]:
        """Renders into the CUDA tensor `out` of shape [H, W, 4] on this renderer's device: dtype
        uint8 (RGBA8), float16 (RGBA16F) or float32 (RGBA32F). Its last two dims must be
        contiguous; the row stride is out.stride(0).
        The frame is rendered on torch.cuda.current_stream(device): this sets the renderer's
        stream to it (set_stream), so later calls on this renderer run on that stream too, and
        the tensor is ready for work queued on it afterwards without a synchronisation."""
        import torch  # only this method needs torch

        if not isinstance(out, torch.Tensor) or not out.is_cuda or out.device.index != self.device:
            raise FormaError(f"Renderer::render_tensor: `out` must be a CUDA tensor on cuda:{self.device}")
        dtypes = {torch.uint8: Format.RGBA8, torch.float16: Format.RGBA16F, torch.float32: Format.RGBA32F}
        if out.dtype not in dtypes:
            raise FormaError(f"Renderer::render_tensor: dtype {out.dtype} is not uint8, float16 or float32")
        if out.dim() != 3 or out.shape[2] != 4 or out.shape[0] < 1 or out.shape[1] < 1:
            raise FormaError(f"Renderer::render_tensor: shape {tuple(out.shape)} is not [H, W, 4]")
        if out.stride(2) != 1 or out.stride(1) != 4 or out.stride(0) < 4 * out.shape[1]:
            raise FormaError(f"Renderer::render_tensor: strides {out.stride()} (the last two dims must be contiguous)")
        h, w = int(out.shape[0]), int(out.shape[1])
        self.set_stream(torch.cuda.current_stream(out.device).cuda_stream)
        return self.render_device(composition, out.data_ptr(), w, h, channels, clear_color, crop, layer_cache,
                                  out.stride(0) * out.element_size(), timings, dtypes[out.dtype])

    def launch_count(self) -> int:
        return int(self._api.renderer_launch_count(self._h))

    STAGES = ("upload", "line_setup", "rasterize", "sort", "paint_tables", "paint_kernel", "d2h", "total")

    def stage_times(self) -> dict:
        """Device-timeline ms of the last render, by stage."""
        out = (C.c_double * 8)()
        self._api.renderer_stage_times(self._h, out)
        return dict(zip(self.STAGES, list(out)))

    def kernel_times(self) -> dict:
        """CUDA-event ms and launch counts of single kernels in the last render."""
        ms, n = (C.c_double * 4)(), (C.c_uint32 * 4)()
        self._api.renderer_kernel_times(self._h, ms, n)
        names = ("radix_downsweep", "radix_upsweep_scan", "paint")
        return {k: {"ms": float(ms[i]), "launches": int(n[i])} for i, k in enumerate(names)}

    def counters(self) -> dict:
        out = (C.c_uint64 * 8)()
        self._api.renderer_counters(self._h, out)
        return dict(zip(("launches", "h2d_bytes", "d2h_bytes", "segments", "cells", "entries", "written_tiles",
                         "tables_mode"),  # tables_mode: 0 counts read back, 1 sync-free, 2 sync-free attempt redone
                        [int(v) for v in out]))

    def host_slices(self) -> list:
        """Device-timeline ms of every slice of the last host frame ([] = rendered as one piece)."""
        ms = (C.c_double * 16)()
        n = int(self._api.renderer_host_slices(self._h, ms, None))
        return [float(ms[i]) for i in range(n)]

    def host_slice_stages(self) -> list:
        """Stage times of every slice of the last host frame (dicts keyed like stage_times())."""
        ms, st = (C.c_double * 16)(), (C.c_double * 128)()
        n = int(self._api.renderer_host_slices(self._h, ms, st))
        return [dict(zip(self.STAGES, [float(st[8 * i + k]) for k in range(8)])) for i in range(n)]

    def row_costs(self) -> np.ndarray:
        """Per-tile-row cost of the last render (forma_renderer_row_costs)."""
        n = int(self._api.renderer_row_costs(self._h, 0, None))
        out = np.zeros(n, np.uint64)
        if n:
            self._api.renderer_row_costs(self._h, n, out.ctypes.data_as(_u64p))
        return out

    def set_stream(self, cuda_stream: int) -> None:
        self._api.renderer_set_stream(self._h, C.c_void_p(cuda_stream))

    # stage-level access ----------------------------------------------------
    def lines(self):
        n = int(self._api.renderer_lines(self._h, 0, None, None, None, None, None, None, None, None, None, None))
        orders = np.zeros(n, np.uint32)
        lengths = np.zeros(n, np.uint32)
        fl = [np.zeros(n, np.float32) for _ in range(8)]
        self._api.renderer_lines(self._h, n, orders.ctypes.data_as(_u32p), *[a.ctypes.data_as(_fp) for a in fl],
                                 lengths.ctypes.data_as(_u32p))
        names = ["x0", "y0", "dx", "dy", "a", "b", "c", "d"]
        out = {"orders": orders, "lengths": lengths}
        out.update(dict(zip(names, fl)))
        return out

    def segments(self) -> np.ndarray:
        n = int(self._api.renderer_segments(self._h, 0, None))
        out = np.zeros(n, np.uint64)
        self._api.renderer_segments(self._h, n, out.ctypes.data_as(_u64p))
        return out

    def rasterize_only(self, composition: Composition, width: int, height: int) -> np.ndarray:
        n = int(self._api.renderer_rasterize_only(self._h, composition._h, width, height, 0, None))
        out = np.zeros(n, np.uint64)
        self._api.renderer_rasterize_only(self._h, composition._h, width, height, n, out.ctypes.data_as(_u64p))
        return out

    def sort_u64(self, keys: np.ndarray) -> np.ndarray:
        out = np.ascontiguousarray(keys, dtype=np.uint64).copy()
        self._api.check(self._api.renderer_sort_u64(self._h, out.ctypes.data_as(_u64p), out.size), "sort_u64")
        return out

    def __del__(self):
        try:
            self._api.renderer_free(self._h)
        except Exception:
            pass


class MultiRenderer:
    """One renderer over several GPUs of the box (forma_renderer_multi_*): `render` /
    `render_device` have Renderer's arguments minus the layer cache; the frame is split into
    cost-balanced bands of tile rows, one per device."""

    def __init__(self, api: Api, devices: Sequence[int]):
        self._api = api
        arr = (C.c_int * len(devices))(*devices)
        self._h = api.renderer_multi_new(arr, len(devices))
        if not self._h:
            raise FormaError(f"MultiRenderer::new failed: {api.last_error().decode()}")
        self.n = int(api.renderer_multi_device_count(self._h))

    def _call(self, fn, what, composition, ptr, width, height, channels, clear_color, crop, stride, fmt=Format.RGBA8):
        stride = width * Format.BYTES_PER_PIXEL[fmt] if stride is None else stride
        ch = (C.c_uint32 * 4)(*channels)
        cc = (C.c_float * 4)(clear_color.r, clear_color.g, clear_color.b, clear_color.a)
        rect = _CRect(crop.horizontal[0], crop.horizontal[1], crop.vertical[0], crop.vertical[1]) if crop is not None else None
        t = _CTimings()
        head = (self._h, composition._h, ptr) + ((fmt,) if fmt != Format.RGBA8 else ())
        st = fn(*head, width, stride, height, ch, cc, C.byref(rect) if rect is not None else None, C.byref(t))
        self._api.check(st, what)
        return Timings(t.line_setup_ms, t.rasterize_ms, t.sort_ms, t.paint_ms, t.n_lines, t.n_segments)

    def render(self, composition: "Composition", buffer: np.ndarray, width: int, height: int, channels=RGBA,
               clear_color: Color = Color(1.0, 1.0, 1.0, 1.0), crop: Optional[Rect] = None, stride: Optional[int] = None) -> Timings:
        """The buffer's dtype picks the format as in Renderer.render."""
        fmt = Format.of_dtype(buffer.dtype)
        s = width * Format.BYTES_PER_PIXEL[fmt] if stride is None else stride
        assert buffer.flags["C_CONTIGUOUS"] and buffer.nbytes >= height * s
        fn = (self._api.renderer_multi_render if fmt == Format.RGBA8
              else self._api.format_call("renderer_multi_render_format", "MultiRenderer::render"))
        return self._call(fn, "MultiRenderer::render", composition, buffer.ctypes.data_as(C.c_void_p), width, height, channels,
                          clear_color, crop, stride, fmt)

    def render_device(self, composition: "Composition", device_ptr: int, width: int, height: int, channels=RGBA,
                      clear_color: Color = Color(1.0, 1.0, 1.0, 1.0), crop: Optional[Rect] = None,
                      stride: Optional[int] = None, format: int = Format.RGBA8) -> Timings:
        if format not in Format.BYTES_PER_PIXEL:
            raise FormaError(f"MultiRenderer::render_device: unknown format {format}")
        fn = (self._api.renderer_multi_render_device if format == Format.RGBA8
              else self._api.format_call("renderer_multi_render_device_format", "MultiRenderer::render_device"))
        return self._call(fn, "MultiRenderer::render_device", composition, C.c_void_p(device_ptr), width, height, channels,
                          clear_color, crop, stride, format)

    def bands(self):
        """(tile-row boundaries of the next frame's bands, ms of every band in the last frame)."""
        b = (C.c_uint32 * (self.n + 1))()
        ms = (C.c_double * self.n)()
        self._api.renderer_multi_bands(self._h, b, ms)
        return list(b), list(ms)

    def __del__(self):
        try:
            self._api.renderer_multi_free(self._h)
        except Exception:
            pass


# ---------------------------------------------------------------------------
# PixelSegment bit layout helpers (forma/src/cpu/pixel_segment.rs:100-138)
# ---------------------------------------------------------------------------


def unpack_segments(segs: np.ndarray):
    s = segs.astype(np.uint64)
    cover = ((s & np.uint64(0x3F)).astype(np.int64) ^ 0x20) - 0x20
    dam = ((s >> np.uint64(6)) & np.uint64(0x3F)).astype(np.int64)
    return {
        "tile_y": ((s >> np.uint64(53)) & np.uint64(0x7FF)).astype(np.int64) - 1,
        "tile_x": ((s >> np.uint64(41)) & np.uint64(0xFFF)).astype(np.int64) - 1,
        "layer_id": ((s >> np.uint64(20)) & np.uint64(0x1FFFFF)).astype(np.int64),
        "local_x": ((s >> np.uint64(16)) & np.uint64(0xF)).astype(np.int64),
        "local_y": ((s >> np.uint64(12)) & np.uint64(0xF)).astype(np.int64),
        "double_area": dam * cover,
        "cover": cover,
    }
