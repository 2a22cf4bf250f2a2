"""bench.py's output contract, checked on the CPU through the reference arm (`--impl
reference` times the oracle, the one other place that may execute oracle/), and the
refusal of the CUDA arm to run without a device."""
import json
import os
import socket
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def json_lines(text):
    out = []
    for line in text.splitlines():
        line = line.strip()
        if line.startswith("{") and line.endswith("}"):
            out.append(json.loads(line))
    return out


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def check_reference_line(d, n_gpus, steps):
    assert d["impl"] == "reference"
    assert d["metric"] == "frames/sec" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == n_gpus and d["steps"] == steps and d["warmup"] >= 3
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1000.0) < 1.0
    assert d["vs_baseline"] is None and d["config"]["workload"] == "smoke" and d["workload_stats"]["pixel_segments"] > 0
    # `config` and `data` are what the driver compares between the two arms: only keys both arms can fill alike
    assert set(d["config"]) == {"workload", "desc", "width", "height", "l2", "parallelism"} and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["cores"] <= cb["usable_cpus"] and cb["thread_candidates_ms"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "smoke" in cb["sample"]
    assert set(cb["stage_ms"]) == {"line_setup", "rasterize", "sort", "paint"}
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_prints_one_contract_line():
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--workload", "smoke", "--steps", "3", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = json_lines(p.stdout)
    assert len(lines) == 1
    check_reference_line(lines[0], 1, 3)


def test_reference_arm_under_torchrun_only_rank0_works():
    """Launched like the driver launches N > 1: rank 0 alone runs and prints, the other rank exits 0."""
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), BENCH, "--impl", "reference", "--gpus", "2", "--workload", "smoke", "--steps", "2",
           "--warmup", "3"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = json_lines(p.stdout)
    assert len(lines) == 1
    check_reference_line(lines[0], 2, 2)


def oracle_smoke_frame():
    import numpy as np

    from forma_b200.binding import RGBA, Color
    from oracle import oracle
    from workloads import build_scene
    api = oracle.load()
    comp, w, h = build_scene(api, "smoke")
    buf = np.zeros(w * h * 4, np.uint8)
    api.Renderer().render(comp, buf, w, h, RGBA, Color(1.0, 1.0, 1.0, 0.0))
    return buf.reshape(-1, 4).astype(np.float32)


def check_dump(path, names):
    import numpy as np
    index = np.load(path / "pixel_index.npy")
    assert index.dtype == np.float64 and np.array_equal(index, np.arange(640 * 360))
    want = oracle_smoke_frame()
    for name in names:
        got = np.load(path / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, want), name
    assert sorted(p.name for p in path.iterdir()) == sorted(["pixel_index.npy"] + [f"{n}.npy" for n in names])


def test_reference_arm_dumps_its_last_frame(tmp_path):
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--workload", "smoke", "--steps", "2",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    check_reference_line(json_lines(p.stdout)[0], 1, 2)
    check_dump(tmp_path / "out", ["frame_host"])


@pytest.mark.gpu
def test_cuda_arm_dumps_the_frames_of_its_last_timed_step(tmp_path):
    p = subprocess.run([sys.executable, BENCH, "--workload", "smoke", "--steps", "2", "--no-cpu",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json_lines(p.stdout)[0]
    assert d["steps"] == 2 and len(d["step_ms_trace"]) == 2
    check_dump(tmp_path / "out", ["frame_device", "frame_host"])


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--workload", "smoke", "--steps", "0"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "--steps" in p.stderr and not json_lines(p.stdout)


def test_cuda_arm_refuses_to_run_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, BENCH, "--workload", "smoke", "--steps", "1"], capture_output=True, text=True, timeout=300,
                       cwd=ROOT)
    assert p.returncode != 0 and "no CPU fallback" in p.stderr
    assert not json_lines(p.stdout)
