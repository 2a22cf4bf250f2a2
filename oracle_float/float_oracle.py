"""FLOAT-FRAME ORACLE — test infrastructure only.

Loads oracle_float/libforma_float_oracle.so (built by oracle_float/Makefile): the CPU oracle of
oracle/ together with the RGBA16F / RGBA32F output formats (fo_renderer_render_format), through
the same binding classes as the product library. Renderer.render of this API takes uint8,
float16 and float32 host buffers like the product's.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from forma_b200 import binding
from oracle import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libforma_float_oracle.so")
_api = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB):
        subprocess.check_call(["make", "-C", _HERE] + (["-B"] if force else []))
    return _LIB


def load() -> binding.Api:
    """The API of the float-frame oracle (cached: its hooks are declared once)."""
    global _api
    if _api is None:
        lib = C.CDLL(build())
        # What the oracle may lack stays optional; the float-frame call is required.
        base = oracle.load()
        optional = [n for n in binding.SIGNATURES if n != "renderer_render_format" and not hasattr(base.lib, "fo_" + n)]
        api = binding.Api(lib, "fo_", optional=optional)
        oracle._declare_hooks(lib)
        f, u32, u64 = C.c_float, C.c_uint32, C.c_uint64
        lib.fo_encode_srgb.restype, lib.fo_encode_srgb.argtypes = None, [C.POINTER(f), u64, C.POINTER(u32), C.POINTER(C.c_uint8)]
        lib.fo_f32_to_f16.restype, lib.fo_f32_to_f16.argtypes = None, [C.POINTER(f), u64, C.POINTER(C.c_uint16)]
        api.hooks = lib
        _api = api
    return _api


def encode_srgb(frame, channels):
    """sRGB bytes of a float32 frame (..., 4) rendered with `channels` (Alpha already One where the
    clear colour is opaque): the RGBA8 frame's values."""
    lib = load().hooks
    f = np.ascontiguousarray(frame, np.float32)
    out = np.zeros(f.shape, np.uint8)
    ch = (C.c_uint32 * 4)(*channels)
    lib.fo_encode_srgb(f.ctypes.data_as(C.POINTER(C.c_float)), f.size // 4, ch, out.ctypes.data_as(C.POINTER(C.c_uint8)))
    return out


def f32_to_f16(values):
    """The oracle's RGBA16F conversion of float32 values (round to nearest even), as float16."""
    lib = load().hooks
    v = np.ascontiguousarray(values, np.float32)
    out = np.zeros(v.shape, np.uint16)
    lib.fo_f32_to_f16(v.ctypes.data_as(C.POINTER(C.c_float)), v.size, out.ctypes.data_as(C.POINTER(C.c_uint16)))
    return out.view(np.float16)
