#!/usr/bin/env python
"""Benchmark of the hot path: one `Renderer::render` of a synthetic or
fixture-backed Composition per step (BASELINE.json metric: frames/s and
pixel-segments/s).

    python bench.py --gpus N --steps K --warmup W [--workload paris4k|cubics100k|circles8k] [--impl reference]

One JSON line on stdout (rank 0). Keys follow the driver's contract:
  value        frames/s with the composition resident in HBM and the frame left
               in HBM (render_device), device-timed, L2 flushed between steps
  e2e          frames/s through the public call with HOST buffers: every step
               re-uploads the whole composition from pinned host memory
               (Composition.evict) and copies the frame back to pinned host memory
  roofline     dominant kernel group: algorithmic bytes / its CUDA-event time
  cpu_baseline the CPU oracle ("forma CPU path, restated") on the host cores
`--impl reference` times that CPU restatement as its own arm (the Rust crate
cannot be built here: no cargo/rustc, see DESIGN.md).

`--dump-outputs DIR` writes the frames of the headline workload's last timed step (CUDA arm:
frame_device.npy from render_device, frame_host.npy from the host-buffer call; reference arm:
frame_host.npy) with pixel_index.npy, so that two builds can be compared pixel for pixel: the
scenes are seeded, so the same arguments give the same inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from workloads import WORKLOADS, build_scene  # noqa: E402  (tests/workloads.py: shared with the parity tests)


def config_of(args, world):
    """Identical in both arms (the driver compares the two `config` dicts)."""
    w, h, desc = WORKLOADS[args.workload]
    return {"workload": args.workload, "desc": desc, "width": w, "height": h,
            "l2": "CUDA arm: L2 flushed between steps (384 MiB memset, untimed)", "parallelism": f"tile-band x{world}"}


def data_of(args):
    return "paris-30k fixture" if args.workload.startswith("paris4k") else "synthetic"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def init_nvml(self):
        """NVML in-process, queried by sample_now() between the timed steps (inside the
        timed region as a whole, while the GPU runs the untimed L2 flush): polling NVML
        from a second thread while render() runs can stall CUDA calls for milliseconds."""
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.hd = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.mx = pynvml.nvmlDeviceGetMaxClockInfo(self.hd, pynvml.NVML_CLOCK_SM)
            self.bits = [pynvml.nvmlClocksThrottleReasonHwSlowdown, pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                         pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, pynvml.nvmlClocksThrottleReasonSwPowerCap]
            return True
        except Exception:
            self.nv = None
            return False

    def sample_now(self):
        if not getattr(self, "nv", None):
            return
        try:
            sm = self.nv.nvmlDeviceGetClockInfo(self.hd, self.nv.NVML_CLOCK_SM)
            r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.hd)
            self.samples.append([str(sm), str(self.mx), "0"] + ["Active" if r & b else "Not Active" for b in self.bits])
        except Exception:
            pass

    def run(self):
        if getattr(self, "nv", None):
            return  # NVML: sampled synchronously by sample_now()
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([v.strip() for v in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def usable_cpus():
    """Hardware threads this process may really use: the affinity mask, capped by the
    cgroup CPU quota (a container on a 256-thread host is often allowed far fewer)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                n = min(n, max(1, int(float(quota) / period)))
            break
        except Exception:
            continue
    return max(1, n)


def tune_cpu_threads(api, render_once, frames=3):
    """The CPU port scales poorly past the physical cores / one NUMA node on some hosts:
    try a few OpenMP thread counts and keep the best, so the baseline uses "all the host
    threads it can use" to its advantage. Every candidate renders one warm-up frame and then
    `frames` timed frames; its score is the fastest of them (a single frame is too noisy: round
    1's two CPU legs picked 64 and 16 threads on the same box and differed 2.6x). Candidates
    never exceed what the affinity mask / cgroup quota allows."""
    ncpu = usable_cpus()
    cands = sorted({c for c in (4, 8, 16, 24, 32, 48, 64, 96, 128, 192, 256, ncpu, ncpu // 2, (3 * ncpu) // 4)
                    if 1 <= c <= ncpu})
    table, best, best_dt = {}, cands[-1], float("inf")
    for c in cands:
        api.hooks.fo_set_num_threads(c)
        render_once()
        dts = []
        for _ in range(frames):
            t0 = time.perf_counter()
            render_once()
            dts.append(time.perf_counter() - t0)
        table[c] = round(1e3 * min(dts), 2)
        if min(dts) < best_dt:
            best, best_dt = c, min(dts)
        if min(dts) > 4.0 * best_dt:  # far off the best already: larger counts will not recover
            break
    api.hooks.fo_set_num_threads(best)
    return best, ncpu, table


def cpu_leg(workload, steps, warmup, budget_s=None):
    """The CPU oracle (port of forma's CPU path, oracle/) rendering `workload` on the host
    cores: thread count tuned first, then `warmup` untimed and up to `steps` timed frames
    (stopping early once `budget_s` seconds are spent). Only render() calls are timed: the
    layer updates of animated workloads are untimed on both arms. Returns the numbers and
    the last frame (for the frame_matches_oracle check)."""
    from forma_b200.binding import RGBA, Color
    from oracle import oracle
    api = oracle.load()
    comp, w, h = build_scene(api, workload)
    r = api.Renderer()
    buf = np.zeros(w * h * 4, np.uint8)
    clear = Color(1.0, 1.0, 1.0, 0.0)
    animate = getattr(comp, "animate", None)
    cache = r.create_buffer_layer_cache() if animate else None
    frame_no, spent = [0], [0.0]

    def one_frame():
        if animate:
            frame_no[0] += 1
            animate(frame_no[0])
        t_in = time.perf_counter()
        t = r.render(comp, buf, w, h, RGBA, clear, None, cache)
        spent[0] += time.perf_counter() - t_in
        return t
    best, ncpu, table = tune_cpu_threads(api, one_frame)
    for _ in range(warmup):
        one_frame()
    n, t0, stages, spent[0] = 0, time.perf_counter(), np.zeros(4), 0.0
    t = None
    while n < steps and (budget_s is None or n == 0 or time.perf_counter() - t0 < budget_s):
        t = one_frame()
        stages += [t.line_setup_ms, t.rasterize_ms, t.sort_ms, t.paint_ms]
        n += 1
    dt = spent[0]
    return {"fps": n / dt, "ms_per_step": 1e3 * dt / n, "frames": n, "cores": api.hooks.fo_num_threads(), "usable_cpus": ncpu,
            "thread_candidates_ms": table, "n_segments": int(t.n_segments), "frame": buf, "frame_no": frame_no[0],
            "stage_ms": dict(zip(["line_setup", "rasterize", "sort", "paint"], (stages / n).round(3).tolist()))}


def cpu_baseline_block(leg, workload, warmup):
    return {"value": leg["fps"], "unit": "frames/s", "cores": leg["cores"], "usable_cpus": leg["usable_cpus"], "kind": "port",
            "sample": f"{leg['frames']} full frames of {workload} after {warmup} warm-up frames",
            "thread_candidates_ms": leg["thread_candidates_ms"], "stage_ms": leg["stage_ms"]}


def run_reference(args):
    """CPU arm: the oracle (port of forma's CPU path) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    leg = cpu_leg(args.workload, args.steps, args.warmup)
    if args.dump_outputs:
        w, h, _ = WORKLOADS[args.workload]
        dump_outputs(args.dump_outputs, {"frame_host": leg["frame"]}, w, h)
    fps = leg["fps"]
    out = {
        "impl": "reference", "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32+f64/u64", "data": data_of(args),
        "config": config_of(args, args.gpus),
        "workload_stats": {"pixel_segments": leg["n_segments"]},
        "mpixel_segments_per_s": leg["n_segments"] * fps / 1e6,
        "cpu_baseline": cpu_baseline_block(leg, args.workload, args.warmup),
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    extra = extra_workloads(args)
    if extra:
        out["extra"] = {}
        for name in extra:
            # A bounded sample: the 8K scene takes seconds per frame on the CPU.
            e = cpu_leg(name, min(args.steps, 3), 1, budget_s=60.0)
            out["extra"][name] = {"value": e["fps"], "unit": "frames/s", "ms_per_step": e["ms_per_step"],
                                  "e2e": {"value": e["fps"], "unit": "frames/s"}, "pixel_segments": e["n_segments"],
                                  "cpu_baseline": cpu_baseline_block(e, name, 1)}
    print(json.dumps(out))


def extra_workloads(args):
    """Scenes timed in addition to the headline workload and printed under "extra": the
    north_star's scaling scene (BASELINE config 5) rides along with every --gpus N run so that
    the driver's 1/2/4/8 sweep records its curve too, while `value` stays the headline scene."""
    if args.extra is None:
        return ["circles8k_1m"] if args.workload == "paris4k" and not args.no_extra else []
    return [w for w in args.extra.split(",") if w]


class SharedHostFrame:
    """One frame in host memory that every rank of the box can write: a /dev/shm file mapped
    by all ranks and page-locked in each of them (cudaHostRegister), so that every GPU copies
    its own band of tile rows straight to its place in the frame (sharded device->host copy).
    With one rank it is an ordinary pinned buffer."""

    def __init__(self, torch, dist, nbytes, rank, world, tag):
        import mmap
        self.torch, self.path, self.registered = torch, None, False
        if world == 1:
            self.tensor = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            self.np = self.tensor.numpy()
            return
        box = [None]
        if rank == 0:
            box[0] = f"/dev/shm/forma_b200_{os.getpid()}_{tag}"
            with open(box[0], "wb") as f:
                f.truncate(nbytes)
        dist.broadcast_object_list(box, src=0)
        self.path = box[0]
        self.file = open(self.path, "r+b")
        self.map = mmap.mmap(self.file.fileno(), nbytes)
        self.np = np.frombuffer(self.map, dtype=np.uint8)
        try:  # page-lock the mapping in this process; pageable memory still works, just slower
            rc = torch.cuda.cudart().cudaHostRegister(self.np.ctypes.data, nbytes, 0)
            self.registered = (int(rc) == 0) if not isinstance(rc, tuple) else (int(rc[0]) == 0)
        except Exception:
            self.registered = False
        dist.barrier()
        if rank == 0:
            os.unlink(self.path)  # the mappings keep it alive

    def close(self):
        if self.path is None:
            return
        try:
            if self.registered:
                self.torch.cuda.cudart().cudaHostUnregister(self.np.ctypes.data)
        except Exception:
            pass


def bench_workload(env, args, name, steps, warmup, headline):
    """Times `name` at env.world GPUs. Returns the result dict on rank 0 (None elsewhere)."""
    torch, dist, api = env["torch"], env["dist"], env["api"]
    rank, world, local, dev, stream, sampler = env["rank"], env["world"], env["local"], env["dev"], env["stream"], env["sampler"]
    from forma_b200 import bands
    from forma_b200.binding import RGBA, Color, Rect

    t_build = time.perf_counter()
    comp, w, h = build_scene(api, name)
    t_build = time.perf_counter() - t_build
    renderer = api.Renderer(local)
    renderer.set_stream(stream.cuda_stream)
    clear = Color(1.0, 1.0, 1.0, 0.0)
    stride = w * 4
    animate = getattr(comp, "animate", None)
    frame_no = [0]

    def next_frame():
        if animate:
            frame_no[0] += 1
            animate(frame_no[0])

    # Tile-row bands. With several GPUs every rank first renders the whole frame once
    # (untimed) and reads the per-tile-row cost of that frame; the band boundaries are
    # then chosen so that every rank gets the same share of that cost (SURVEY.md 8e).
    # The cost table is a deterministic function of the scene, identical on all ranks.
    fb = torch.zeros((h, stride), dtype=torch.uint8, device=dev)
    balance = "single"
    bd = bands.band_of(h, world, rank)
    if world > 1:
        next_frame()
        renderer.render_device(comp, fb.data_ptr(), w, h, RGBA, clear, None, None, stride)
        torch.cuda.synchronize()
        costs = renderer.row_costs() if hasattr(renderer, "row_costs") else None
        if costs is not None and len(costs) and not args.equal_bands:
            # + a floor per row: every tile of a row is at least cleared and stored
            costs = [float(c) + 2.0 * ((w + 15) // 16) for c in costs]
            bd = bands.balanced_band(h, world, rank, costs)
            balance = "previous frame's per-row cost"
        else:
            balance = "equal rows"
        comp.evict()  # from here on this rank only keeps its band's geometry resident
    r0, r1 = bd.tile_row0, bd.tile_row1
    crop = None if world == 1 else Rect((0, w), (bd.y0, max(bd.y1, bd.y0)))
    host = SharedHostFrame(torch, dist, h * stride, rank, world, name)
    host_np = host.np

    gather_events = []
    # Frame assembly over NVLink: rank 0 owns the frame, the other ranks map it (CUDA IPC)
    # and their paint kernels store their bands straight into rank 0's HBM; a 1-element NCCL
    # all-reduce on the render streams closes the frame. Fallback (IPC unavailable): every
    # rank paints locally and rank 0 receives the bands with NCCL send/recv.
    shared, frame_ptr, flag, whole = None, fb.data_ptr(), None, None
    assembly = None
    if world > 1:
        assembly = "p2p"
        nbytes = h * stride
        box, ok = [None], 1.0
        try:
            if rank == 0:
                shared = api.SharedFrame(local, nbytes)
                box = [shared.handle]
        except Exception:
            ok = 0.0
        dist.broadcast_object_list(box, src=0)
        try:
            if rank != 0 and box[0] is not None:
                shared = api.SharedFrame(local, nbytes, box[0])
        except Exception:
            ok = 0.0
        if shared is None:
            ok = 0.0
        flag = torch.tensor([ok], dtype=torch.float32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if float(flag.item()) >= 1.0:
            frame_ptr = shared.ptr
            if rank == 0:
                whole = torch.as_tensor(shared, device=dev).view(h, stride)
        else:
            shared, assembly = None, "sendrecv"
            if rank == 0:
                whole = fb
        flag = torch.zeros(1, dtype=torch.float32, device=dev)  # the per-frame closing all-reduce works on this
        all_bands = [bands.balanced_band(h, world, r, costs) if balance.startswith("previous") else bands.band_of(h, world, r)
                     for r in range(world)]

    # Animated workloads render with a persistent layer cache (one per target buffer, like the
    # reference's per-Buffer caches).
    cache_dev = renderer.create_buffer_layer_cache() if animate else None
    cache_host = renderer.create_buffer_layer_cache() if animate else None

    def frame_device():
        renderer.render_device(comp, frame_ptr, w, h, RGBA, clear, crop, cache_dev, stride, timings=False)
        if world > 1:
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            if shared is not None:
                dist.all_reduce(flag)
            else:
                if rank == 0:
                    for b in all_bands[1:]:
                        if b.y1 > b.y0:
                            dist.recv(fb[b.y0:b.y1], src=b.rank)
                elif bd.y1 > bd.y0:
                    dist.send(fb[bd.y0:bd.y1], dst=0)
            g1.record(stream)
            gather_events.append((g0, g1))

    def frame_e2e():
        # The public host-buffer call: the composition is re-uploaded from pinned host memory
        # (evict) and the frame (this rank's band) is copied back to (its place in) the host
        # frame, all inside the timed region.
        comp.evict()
        renderer.render(comp, host_np, w, h, RGBA, clear, crop, cache_host, stride, timings=False)

    flush = env["flush"]

    def timed(fn, n, after=None):
        """Per-step CUDA events on the launching stream; the L2 flush runs between steps, untimed.
        `after` (reading the step's stage times: a dozen event queries) runs behind the step's
        closing synchronisation, outside the timed interval - it is diagnostics, not rendering."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        wall = 0.0
        for a, b in evs:
            flush.zero_()
            sampler.sample_now()  # SM clock / throttle reasons while the GPU is busy, outside the timed interval
            # Animated workloads: the layer updates of the next frame are host-side API calls;
            # they run here, outside the timed region, on both arms.
            next_frame()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize()
            wall += time.perf_counter() - t0  # all ranks start together (barrier above); the frame is complete after the slowest one (max over ranks below)
            if after:
                after()
        dev_ms = sum(a.elapsed_time(b) for a, b in evs)
        return dev_ms, wall * 1e3

    for _ in range(max(warmup, 1)):
        next_frame()
        frame_device()
    torch.cuda.synchronize()
    assembled_ok = None
    if world > 1:  # untimed check: the assembled frame equals rank 0's own single-GPU frame, byte for byte
        dist.barrier()
        if rank == 0:
            ref = torch.zeros((h, stride), dtype=torch.uint8, device=dev)
            renderer.render_device(comp, ref.data_ptr(), w, h, RGBA, clear, None, None, stride)
            torch.cuda.synchronize()
            assembled_ok = bool(torch.equal(ref[:, :w * 4], whole[:h, :w * 4]))
            del ref
            comp.evict()  # the whole-frame render made everything resident again: back to the band
        dist.barrier()
        frame_device()
        torch.cuda.synchronize()
    c0 = renderer.counters()
    stage_acc = {k: 0.0 for k in renderer.STAGES}
    kern_acc, step_trace = {}, []

    def device_acc():
        st = renderer.stage_times()
        step_trace.append(round(st["total"], 3))
        for k, v in st.items():
            stage_acc[k] += v
        for k, v in renderer.kernel_times().items():
            a = kern_acc.setdefault(k, {"ms": 0.0, "launches": 0})
            a["ms"] += v["ms"]
            a["launches"] += v["launches"]
    dev_ms, wall_ms = timed(frame_device, steps, device_acc)
    c1 = renderer.counters()
    # The device-resident frame of the last timed step, for --dump-outputs (rank 0 holds the whole frame);
    # kept on the device until the timing below is over.
    device_frame = (whole if world > 1 else fb).clone() if headline and args.dump_outputs and rank == 0 else None
    gather_ms = sum(a.elapsed_time(b) for a, b in gather_events[-steps:]) / steps if gather_events else 0.0
    render_ms = stage_acc["total"] / steps
    for _ in range(max(warmup, 1)):
        next_frame()
        frame_e2e()
    c2 = renderer.counters()
    e2e_stage_acc = {k: 0.0 for k in renderer.STAGES}

    def e2e_acc():
        for k, v in renderer.stage_times().items():
            e2e_stage_acc[k] += v
    e2e_dev_ms, e2e_wall_ms = timed(frame_e2e, steps, e2e_acc)
    c3 = renderer.counters()
    slice_ms = renderer.host_slices() if hasattr(renderer, "host_slices") else []

    def reduce_ranks(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())
    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM) if world > 1 else (None, None)

    # The render call blocks on small device->host count read-backs, so wall time and the
    # device timeline agree; report the slower of the two, max over ranks.
    gather_ms_max = reduce_ranks(gather_ms, MAX)  # includes waiting for the slowest rank's band
    render_ms_max, render_ms_min = reduce_ranks(render_ms, MAX), -reduce_ranks(-render_ms, MAX)
    T = reduce_ranks(max(dev_ms, wall_ms), MAX)
    T_e2e = reduce_ranks(max(e2e_dev_ms, e2e_wall_ms), MAX)
    n_seg = c1["segments"]
    n_seg_total = int(reduce_ranks(float(n_seg), SUM))
    h2d_total = int(reduce_ranks(float(c3["h2d_bytes"] - c2["h2d_bytes"]), SUM)) // steps  # counted by the library, all ranks
    d2h_total = int(reduce_ranks(float(c3["d2h_bytes"] - c2["d2h_bytes"]), SUM)) // steps
    launches_e2e = int(reduce_ranks(float(c3["launches"] - c2["launches"]), SUM))
    launches_dev = int(reduce_ranks(float(c1["launches"] - c0["launches"]), SUM))
    stage_rows = None
    if world > 1:  # every rank's stage times, for the scaling analysis
        mine = torch.tensor([stage_acc[k] / steps for k in renderer.STAGES], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        stage_rows = [[round(float(x), 4) for x in r.tolist()] for r in allr]
    frame_copy = host_np.copy() if rank == 0 else None
    host.close()
    if rank != 0:
        return None

    fps = steps / (T / 1e3)
    fps_e2e = steps / (T_e2e / 1e3)
    stages = {k: v / steps for k, v in stage_acc.items()}
    peak, peak_kind = measured_peak_gbs()
    # Dominant kernel (rank 0): the one with the largest time per step among the radix
    # downsweep, the radix upsweep + scan and the paint kernel, timed per launch with CUDA
    # events on the launching stream inside Renderer::render.
    band_px = (min(r1 * 16, h) - r0 * 16) * w
    # Per-launch algorithmic bytes (DESIGN.md): a radix downsweep launch reads and writes every
    # key once (16 N), an upsweep launch reads them once (8 N), the paint kernel reads the
    # segments and writes the framebuffer once (8 N + 4 W H).
    per_launch = {"radix_downsweep": 16.0 * n_seg, "radix_upsweep_scan": 8.0 * n_seg,
                  "paint": 8.0 * n_seg + 4.0 * band_px}
    kerns = {}
    for k, a in kern_acc.items():
        if a["launches"] and a["ms"] > 0:
            avg_ms = a["ms"] / a["launches"]
            kerns[k] = {"ms_per_launch": avg_ms, "launches_per_step": a["launches"] / steps,
                        "ms_per_step": a["ms"] / steps, "algorithmic_bytes_per_launch": per_launch[k],
                        "GBps": per_launch[k] / (avg_ms * 1e-3) / 1e9}
    if "paint" in kerns:  # SURVEY.md 8(d): the painter is not bandwidth-shaped; its own unit is pixel*layers/s
        kerns["paint"]["gpx_layers_per_s"] = c1["entries"] * 256.0 / (kerns["paint"]["ms_per_launch"] * 1e-3) / 1e9
    kname = max(kerns, key=lambda k: kerns[k]["ms_per_step"]) if kerns else None
    dom = kerns.get(kname, {"GBps": 0.0, "ms_per_launch": 0.0, "algorithmic_bytes_per_launch": 0.0})
    sort_ms = stages["sort"]
    # dram__bytes_read + dram__bytes_write of one launch of that kernel, from the committed
    # `ncu --set full` capture of this command (profiles/ncu_traffic.json), or null.
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get(name, {}).get(kname)
    except Exception:
        pass
    roofline = {"kernel": kname, "bound": "hbm", "achieved": dom["GBps"], "peak": peak, "peak_source": peak_kind,
                "unit": "GB/s", "frac": dom["GBps"] / peak, "traffic": traffic,
                "algorithmic_bytes": dom["algorithmic_bytes_per_launch"], "kernel_ms": dom["ms_per_launch"],
                "kernels": kerns,
                # The whole sort against its algorithm-independent bound (SURVEY.md 8d: 16 N).
                "sort_stage": {"ms": sort_ms, "GBps_vs_16N": (16.0 * n_seg / (sort_ms * 1e-3) / 1e9) if sort_ms > 0 else 0.0,
                               "frac_vs_16N": (16.0 * n_seg / (sort_ms * 1e-3) / 1e9 / peak) if sort_ms > 0 else 0.0}}
    out = {
        "value": fps, "unit": "frames/s", "ms_per_step": T / steps,
        "workload_stats": {"pixel_segments": n_seg_total, "points": comp.point_count(), "cells": c1["cells"],
                           "entries": c1["entries"], "scene_build_s": round(t_build, 2)},
        "mpixel_segments_per_s": n_seg_total * fps / 1e6,
        "stage_ms": {k: round(v, 4) for k, v in stages.items()},
        "step_ms_trace": step_trace,  # device-timeline ms of every timed step (a one-off hiccup shows here)
        "gpu_launches": launches_dev,
        "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": T_e2e / steps,
                "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total, "bytes_counted_by": "the library, summed over ranks",
                "gpu_launches": launches_e2e, "host_frame": "pinned" if world == 1 else ("shared, page-locked per rank" if host.registered else "shared, pageable"),
                "stage_ms": {k: round(v / steps, 4) for k, v in e2e_stage_acc.items()},
                # host frames are rendered as a pipeline of tile-row slices (upload / compute / copy-back of
                # neighbouring slices overlap); stage_ms then holds the slowest slice's stages, which overlap the others'
                "host_slices": len(slice_ms), "slice_ms": [round(v, 4) for v in slice_ms]},
        "roofline": roofline,
        "multi_gpu": {"render_ms_slowest_rank": round(render_ms_max, 4), "render_ms_fastest_rank": round(render_ms_min, 4),
                      "assembly": assembly, "bands": balance,
                      "band_rows": [[b.tile_row0, b.tile_row1] for b in all_bands] if world > 1 else None,
                      "assembled_frame_equals_single_gpu_frame": assembled_ok,
                      "assembly_ms": round(gather_ms_max, 4), "frame_bytes": (h * stride) if world > 1 else 0,
                      "stage_ms_per_rank": stage_rows, "stage_names": list(renderer.STAGES) if world > 1 else None},
    }
    out["_frame"] = frame_copy
    out["_frame_no"] = frame_no[0]
    out["_device_frame"] = None if device_frame is None else device_frame.cpu().numpy().reshape(-1)
    return out


def dump_outputs(path, frames, w, h, budget=1 << 20):
    """Writes the RGBA8 frames (flat uint8, w * h * 4 bytes each) as float32 (n, 4) arrays of pixel
    values in `path`/<name>.npy, with `pixel_index.npy` (float64, n): the row-major index y * w + x
    of each of those n pixels. Frames of more than `budget` pixels are sampled at the same `budget`
    pixels, drawn with a fixed seed, so that runs with the same arguments dump the same pixels."""
    os.makedirs(path, exist_ok=True)
    n = w * h
    index = np.arange(n) if n <= budget else np.sort(np.random.default_rng(0).choice(n, budget, replace=False))
    np.save(os.path.join(path, "pixel_index.npy"), index.astype(np.float64))
    for name, frame in frames.items():
        np.save(os.path.join(path, f"{name}.npy"), frame.reshape(n, 4)[index].astype(np.float32))


def run_cuda(args):
    import torch
    import torch.distributed as dist

    import forma_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        sys.exit(f"bench.py: --gpus {args.gpus} but WORLD_SIZE is {world}; launch one rank per GPU with "
                 f"`python -m torch.distributed.run --nnodes=1 --nproc-per-node {args.gpus} --master-addr 127.0.0.1 bench.py --gpus {args.gpus} ...`")
    if not torch.cuda.is_available():
        sys.exit("bench.py: no CUDA device. The forma_b200 arm has no CPU fallback; "
                 "`--impl reference` times the CPU restatement of the reference instead.")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    sampler = ClockSampler(local)
    env = {"torch": torch, "dist": dist, "api": forma_b200.load(), "rank": rank, "world": world, "local": local, "dev": dev,
           "stream": torch.cuda.current_stream(), "sampler": sampler,
           "flush": torch.empty(384 << 20, dtype=torch.uint8, device=dev)}  # > 126 MB L2
    sampler.init_nvml()
    sampler.start()
    res = bench_workload(env, args, args.workload, args.steps, args.warmup, True)
    extras = {}
    for name in extra_workloads(args):
        # Fewer steps for the heavy ride-along scene: its frames take tens of milliseconds.
        e = bench_workload(env, args, name, max(3, min(args.steps, 10)), 3, False)
        if e is not None:
            extras[name] = e
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frame, frame_no, device_frame = res.pop("_frame"), res.pop("_frame_no"), res.pop("_device_frame")
    if args.dump_outputs:
        w, h, _ = WORKLOADS[args.workload]
        dump_outputs(args.dump_outputs, {"frame_device": device_frame, "frame_host": frame}, w, h)
    out = {"metric": "frames/sec", "value": res.pop("value"), "unit": res.pop("unit"), "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f32+f64/u64", "data": data_of(args), "config": config_of(args, world)}
    out.update(res)
    out["library_options"] = {k: env["api"].get_option(k) for k in ("sync_free", "speculate", "copy_bands", "host_slices", "band_filter", "paint_lpt")}
    out["clocks"] = sampler.summary()
    if extras:
        out["extra"] = {}
        for name, e in extras.items():
            e.pop("_frame")
            e.pop("_frame_no")
            e.pop("_device_frame")
            e.pop("step_ms_trace", None)
            out["extra"][name] = e
    if world == 1 and not args.no_cpu:
        # The CPU oracle on the host cores, on the same scene: a reported baseline, and the
        # checker of the frame that was just timed (the e2e frame in host memory).
        leg = cpu_leg(args.workload, 40, 2, budget_s=12.0)
        out["cpu_baseline"] = cpu_baseline_block(leg, args.workload, 2)
        if frame is not None:
            if leg["frame_no"] != frame_no:  # animated: bring the oracle to the frame the GPU rendered last
                out["frame_matches_oracle"] = oracle_frame_matches(args.workload, frame_no, frame)
            else:
                out["frame_matches_oracle"] = bool(np.array_equal(leg["frame"], frame))
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def oracle_frame_matches(workload, frame_no, gpu_frame):
    """Renders frame `frame_no` of an animated workload with the oracle (no cache: the cache
    never changes pixels) and compares it with the GPU's host frame."""
    from forma_b200.binding import RGBA, Color
    from oracle import oracle
    api = oracle.load()
    comp, w, h = build_scene(api, workload)
    if getattr(comp, "animate", None):
        comp.animate(frame_no)
    buf = np.zeros(w * h * 4, np.uint8)
    api.Renderer().render(comp, buf, w, h, RGBA, Color(1.0, 1.0, 1.0, 0.0))
    return bool(np.array_equal(buf, gpu_frame))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="paris4k", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--extra", default=None,
                    help="comma-separated workloads timed after the headline one and printed under \"extra\" "
                         "(default: circles8k_1m, BASELINE config 5, when the headline workload is paris4k)")
    ap.add_argument("--no-extra", action="store_true", help="headline workload only")
    ap.add_argument("--equal-bands", action="store_true", help="multi-GPU: equal tile-row bands instead of cost-balanced ones")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the frames of the headline workload's last timed step "
                         "as DIR/<name>.npy (float32 pixel values; frames over 2^20 pixels as a fixed seeded sample of 2^20 pixels)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
