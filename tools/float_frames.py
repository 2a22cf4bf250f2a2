"""Frame rate of the three output formats (RGBA8, RGBA16F, RGBA32F) on one GPU.

    python tools/float_frames.py [--workloads paris4k,cubics100k,circles8k_1m] [--steps 20] [--warmup 3] [--out FILE]

Per workload and format, one JSON line with
  * device_fps: frames/s with the frame in HBM (forma_renderer_render_device_format),
  * e2e_fps: frames/s of the host-buffer call after forma_composition_evict (upload, render,
    copy-back: forma_renderer_render_format),
  * paint_ms: the paint kernel's CUDA-event time of the device frames (forma_renderer_kernel_times),
  * d2h_bytes: device->host bytes per end-to-end frame (counters()["d2h_bytes"]).
Timing follows bench.py: CUDA events around the public call, closed by a synchronise; the L2
(126 MB) overwritten by a 384 MiB memset before every step, untimed; warm-up frames first. The
formats are alternated step by step in one process, so that they share the machine's state.
The GPU's name and power limit are recorded on every line. circles8k_1m is BASELINE config 5
(1 M paths at 7680x4320)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def gpu_info(index: int) -> dict:
    import torch
    info = {"gpu": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(out[0]), float(out[1])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        info["power_limit_w"] = None
    return info


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--workloads", default="paris4k,cubics100k,circles8k_1m")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    import numpy as np
    import torch

    import forma_b200
    import workloads
    from forma_b200.binding import RGBA, Color, Format

    dev = torch.device("cuda", args.device)
    torch.cuda.set_device(dev)
    api = forma_b200.load()
    info = gpu_info(args.device)
    flush = torch.empty(384 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    clear = Color(1.0, 1.0, 1.0, 1.0)
    formats = [("rgba8", Format.RGBA8), ("rgba16f", Format.RGBA16F), ("rgba32f", Format.RGBA32F)]
    lines = []
    for name in args.workloads.split(","):
        comp, w, h = workloads.build_scene(api, name)
        r = api.Renderer(args.device)
        r.set_stream(stream.cuda_stream)
        tdt = {Format.RGBA8: torch.uint8, Format.RGBA16F: torch.float16, Format.RGBA32F: torch.float32}
        dev_frames = {f: torch.empty((h, w, 4), dtype=tdt[f], device=dev) for _, f in formats}
        host_frames = {f: torch.empty((h, w, 4), dtype=tdt[f]).pin_memory().numpy().reshape(-1) for _, f in formats}
        acc = {f: {"device_ms": [], "e2e_ms": [], "paint_ms": [], "d2h_bytes": []} for _, f in formats}

        def device_frame(f):
            r.render_device(comp, dev_frames[f].data_ptr(), w, h, RGBA, clear, timings=False, format=f)

        def e2e_frame(f):
            comp.evict()
            r.render(comp, host_frames[f], w, h, RGBA, clear, timings=False)

        def timed(fn):
            flush.zero_()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize()
            return a.elapsed_time(b)

        for _ in range(max(args.warmup, 1)):
            for _, f in formats:
                device_frame(f)
                e2e_frame(f)
        torch.cuda.synchronize()
        for _ in range(args.steps):
            for _, f in formats:  # alternated step by step
                acc[f]["device_ms"].append(timed(lambda: device_frame(f)))
                acc[f]["paint_ms"].append(r.kernel_times()["paint"]["ms"])
                before = r.counters()["d2h_bytes"]
                acc[f]["e2e_ms"].append(timed(lambda: e2e_frame(f)))
                acc[f]["d2h_bytes"].append(r.counters()["d2h_bytes"] - before)
        for label, f in formats:
            a = acc[f]
            line = {"workload": name, "width": w, "height": h, "format": label, "steps": args.steps, "warmup": args.warmup,
                    "device_fps": round(1e3 * len(a["device_ms"]) / sum(a["device_ms"]), 2),
                    "device_ms_median": round(float(np.median(a["device_ms"])), 4),
                    "e2e_fps": round(1e3 * len(a["e2e_ms"]) / sum(a["e2e_ms"]), 2),
                    "e2e_ms_median": round(float(np.median(a["e2e_ms"])), 4),
                    "paint_ms_median": round(float(np.median(a["paint_ms"])), 4),
                    "d2h_bytes_per_frame": int(np.median(a["d2h_bytes"])),
                    "l2": "384 MiB memset between steps, untimed", **info,
                    "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())}
            lines.append(line)
            print(json.dumps(line), flush=True)
        del comp, r, dev_frames, host_frames
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for line in lines:
                fh.write(json.dumps(line) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
