"""Headless front end: render an SVG file to PPM / PNG on the GPU.

    python -m forma_b200.render in.svg out.ppm [--width W --height H --scale S --device 0]
    python -m forma_b200.render in.svg out.npy --format rgba16f|rgba32f [...]

The equivalent of the reference's `demo svg --file in.svg --scale S` + the `S` key's
capture.ppm (demo/src/main.rs, demo/src/runner.rs:193-219: a binary P6 file with the
frame's RGB bytes), without a window. The output format follows the extension (.ppm, or
.png when Pillow is available); both hold the RGBA8 (sRGB) frame. With --format rgba16f or
rgba32f the frame is the painter's linear colour (what the reference's gpu::Renderer leaves in
its Rgba16Float texture), written as an (H, W, 4) float16 / float32 .npy. There is no CPU
fallback: without a CUDA device the renderer cannot be created and the command fails.
"""
from __future__ import annotations

import argparse
import sys
import time

import numpy as np


def write_ppm(path: str, rgba: np.ndarray, width: int, height: int) -> None:
    """runner.rs:193-219: "P6\\n{w} {h}\\n255\\n" + RGB triples."""
    rgb = np.ascontiguousarray(rgba.reshape(height, width, 4)[:, :, :3])
    with open(path, "wb") as f:
        f.write(f"P6\n{width} {height}\n255\n".encode())
        f.write(rgb.tobytes())


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m forma_b200.render", description=__doc__.split("\n\n")[0])
    ap.add_argument("svg")
    ap.add_argument("out")
    ap.add_argument("--width", type=int, default=1000)   # App::width / height of the demo (svg.rs:860-868)
    ap.add_argument("--height", type=int, default=1000)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--frames", type=int, default=1, help="render this many times and report the last frame's timings")
    ap.add_argument("--format", choices=("rgba8", "rgba16f", "rgba32f"), default="rgba8",
                    help="frame format; rgba16f / rgba32f (linear) need an .npy output")
    args = ap.parse_args(argv)
    if args.format != "rgba8" and not args.out.lower().endswith(".npy"):
        ap.error("--format rgba16f / rgba32f writes a linear frame: the output must be a .npy file")

    import forma_b200
    from forma_b200 import svg
    from forma_b200.binding import RGBA, Color, Format

    t0 = time.perf_counter()
    paths = svg.parse_svg(args.svg)
    t1 = time.perf_counter()
    api = forma_b200.load()
    renderer = api.Renderer(args.device)  # raises without a usable GPU
    comp = api.Composition()
    svg.compose(api, comp, paths, scale=args.scale)
    fmt = Format.NAMES[args.format]
    buf = np.zeros(args.width * args.height * 4, Format.DTYPES[fmt])
    t2 = time.perf_counter()
    for _ in range(max(args.frames, 1)):
        t = renderer.render(comp, buf, args.width, args.height, RGBA, Color(1.0, 1.0, 1.0, 1.0))  # the demo clears to white
    t3 = time.perf_counter()
    if args.out.lower().endswith(".npy"):
        np.save(args.out, buf.reshape(args.height, args.width, 4))
    elif args.out.lower().endswith(".png"):
        from PIL import Image
        Image.fromarray(buf.reshape(args.height, args.width, 4), "RGBA").save(args.out)
    else:
        write_ppm(args.out, buf, args.width, args.height)
    print(f"{len(paths)} paths parsed in {t1 - t0:.2f} s, composed in {t2 - t1:.2f} s; {t.n_segments} pixel segments; "
          f"last frame: line setup {t.line_setup_ms:.3f} ms, rasterize {t.rasterize_ms:.3f} ms, sort {t.sort_ms:.3f} ms, "
          f"paint {t.paint_ms:.3f} ms ({(t3 - t2) / max(args.frames, 1) * 1e3:.2f} ms per call) -> {args.out}", file=sys.stderr)
    return 0


if __name__ == "__main__":
    sys.exit(main())
