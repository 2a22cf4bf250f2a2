"""The SVG subset loader (forma_b200/svg.py, SURVEY.md §8(f) N1) against hand-computed
expectations for every element it handles, against the committed paris-30k fixture, and
through the CPU oracle for a picture-level check of arcs, rectangles and gradients."""
import hashlib
import math
import os

import numpy as np
import pytest

from forma_b200 import svg
from forma_b200.binding import RGBA, BlendMode, Color, GradientType

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

DOC = """<svg xmlns="http://www.w3.org/2000/svg" width="64" height="64">
  <defs>
    <linearGradient id="lg" gradientUnits="userSpaceOnUse" x1="8" y1="0" x2="56" y2="0">
      <stop offset="0%" stop-color="#ff0000"/>
      <stop offset="50%" stop-color="#00ff00" stop-opacity="0.5"/>
      <stop offset="100%" stop-color="#0000ff"/>
    </linearGradient>
    <radialGradient id="rg" gradientUnits="userSpaceOnUse" cx="32" cy="32" r="20">
      <stop offset="0%" stop-color="#ffffff"/>
      <stop offset="100%" stop-color="#000000"/>
    </radialGradient>
    <linearGradient id="ignored" x1="0" y1="0" x2="1" y2="0">
      <stop offset="0%" stop-color="#ff0000"/><stop offset="100%" stop-color="#0000ff"/>
    </linearGradient>
  </defs>
  <rect x="8" y="8" width="48" height="48" fill="url(#lg)"/>
  <g transform="translate(2 3)" fill="#336699" opacity="0.5">
    <path d="M 10 10 h 20 v 20 h -20 z" style="mix-blend-mode: multiply"/>
    <path d="M 30 20 A 10 10 0 0 1 20 30 L 20 20 Z" fill="url(#rg)" fill-rule="evenodd"/>
  </g>
  <path d="M 40 32 a 8 8 0 1 0 16 0 a 8 8 0 1 0 -16 0" fill="#ffffff" fill-opacity="0.25"/>
  <rect x="1" y="1" width="5" height="5" stroke="#000000"/>
</svg>"""


@pytest.fixture(scope="module")
def parsed(tmp_path_factory):
    p = tmp_path_factory.mktemp("svg") / "doc.svg"
    p.write_text(DOC)
    return svg.parse_svg(str(p)), str(p)


def test_elements_commands_and_fills(parsed):
    pl, _ = parsed
    assert len(pl) == 4  # the stroked rect is skipped (svg.rs:701-707)
    # rect: move + four lines, no group transform, gradient fill
    c, q = pl.cmd[pl.cmd_off[0]:pl.cmd_off[1]], pl.pts[pl.pt_off[0]:pl.pt_off[1]]
    assert c.tolist() == [svg.MOVE, svg.LINE, svg.LINE, svg.LINE, svg.LINE]
    assert q.tolist() == [[8, 8], [8, 56], [56, 56], [56, 8], [8, 8]]
    assert pl.grad[0] == 0 and pl.blend[0] == BlendMode.Over
    g = pl.gradients[0]
    assert g["type"] == GradientType.Linear and g["start"] == (8.0, 0.0) and g["end"] == (56.0, 0.0)
    assert [round(s, 6) for _, s in g["stops"]] == [0.0, 0.5, 1.0]
    assert g["stops"][1][0][3] == 0.5 and g["stops"][0][0][:3] == (1.0, 0.0, 0.0)
    # a gradient without userSpaceOnUse is ignored (svg.rs:739-745): only two gradients exist
    assert len(pl.gradients) == 2 and pl.gradients[1]["type"] == GradientType.Radial
    assert pl.gradients[1]["end"] == (52.0, 32.0)  # (cx + r, cy)
    # group: translate applied to points, group fill + opacity, blend mode from style
    q = pl.pts[pl.pt_off[1]:pl.pt_off[2]]
    assert q.tolist() == [[12, 13], [32, 13], [32, 33], [12, 33]]
    assert pl.blend[1] == BlendMode.Multiply and pl.grad[1] == -1
    assert np.allclose(pl.color[1], [svg.to_linear(0x33), svg.to_linear(0x66), svg.to_linear(0x99), 0.5])
    # fill-opacity without opacity; even-odd
    assert pl.color[3][3] == 0.25 and pl.fill_rule[2] == 1 and pl.fill_rule[3] == 0


def test_arc_becomes_rational_quads(parsed):
    pl, _ = parsed
    # path 2: quarter circle of radius 10 around (20, 20) from (30, 20) to (20, 30), then lines
    c = pl.cmd[pl.cmd_off[2]:pl.cmd_off[3]].tolist()
    q = pl.pts[pl.pt_off[2]:pl.pt_off[3]]
    assert c == [svg.MOVE, svg.RATQUAD, svg.LINE]
    assert np.allclose(q[0], [32, 23])                      # translated start
    assert np.allclose(q[1], [32, 33], atol=1e-4)           # control point: the corner of the quarter turn
    assert np.allclose(q[2], [22, 33], atol=1e-4)           # end point
    assert abs(pl.weights[0] - math.cos(math.pi / 4)) < 1e-6
    assert pl.grad[2] == 1
    # path 3: two half circles (large-arc, sweep 0), each split into two quarter turns
    c = pl.cmd[pl.cmd_off[3]:pl.cmd_off[4]].tolist()
    assert c == [svg.MOVE] + [svg.RATQUAD] * 4
    q = pl.pts[pl.pt_off[3]:pl.pt_off[4]]
    assert np.allclose(q[4], [56, 32], atol=1e-4) and np.allclose(q[8], [40, 32], atol=1e-4)
    ws = pl.weights[1:5]
    assert np.allclose(ws, math.cos(math.pi / 4), atol=1e-6)
    # every arc point lies on the circle of radius 8 around (48, 32); control points on its corners
    ends = q[[2, 4, 6, 8]]
    assert np.allclose(np.hypot(ends[:, 0] - 48, ends[:, 1] - 32), 8, atol=1e-3)


def test_convert_to_center_degenerate_cases():
    assert svg.convert_to_center(5, 5, 0, False, True, 1, 1, 1, 1) is None      # coincident end points
    assert svg.convert_to_center(0, 5, 0, False, True, 0, 0, 1, 1) is None      # zero radius
    arc = svg.convert_to_center(1, 1, 0, False, True, 10, 0, -10, 0)            # radii too small: len_squared >= 1, centre = midpoint
    assert arc is not None and abs(arc[0]) < 1e-6 and abs(arc[1]) < 1e-6


def test_pathlist_roundtrip(parsed, tmp_path):
    pl, _ = parsed
    f = tmp_path / "pl.npz"
    pl.save(str(f))
    back = svg.PathList.load(str(f))
    for k in ("cmd", "pts", "cmd_off", "pt_off", "color", "fill_rule", "weights", "blend", "grad"):
        assert np.array_equal(getattr(pl, k), getattr(back, k)), k
    assert back.gradients == pl.gradients


def test_picture_through_the_oracle(parsed, oracle_api):
    """Arcs, rect and gradients end up as the expected picture (CPU oracle; the CUDA path is
    compared with the oracle on the same scenes in the GPU tests)."""
    pl, _ = parsed
    comp = oracle_api.Composition()
    assert svg.compose(oracle_api, comp, pl) == 4
    buf = np.zeros(64 * 64 * 4, np.uint8)
    oracle_api.Renderer(0).render(comp, buf, 64, 64, RGBA, Color(0.0, 0.0, 0.0, 1.0))
    img = buf.reshape(64, 64, 4)
    assert img[4, 4].tolist() == [0, 0, 0, 255]                 # outside everything
    left, right = img[50, 9].astype(int), img[50, 54].astype(int)
    assert left[0] > 200 and left[2] < 40 and right[2] > 200 and right[0] < 40   # the linear gradient runs red -> blue
    # the translucent white disc (two half-circle arcs around (48, 32), r = 8) changes exactly the pixels under it
    comp3 = oracle_api.Composition()
    svg.compose(oracle_api, comp3, pl, limit=3)
    without = np.zeros(64 * 64 * 4, np.uint8)
    oracle_api.Renderer(0).render(comp3, without, 64, 64, RGBA, Color(0.0, 0.0, 0.0, 1.0))
    changed = (img != without.reshape(64, 64, 4)).any(axis=2)
    ys, xs = np.nonzero(changed)
    assert changed[32, 48] and 195 <= changed.sum() <= 240       # pi * 8^2 = 201 pixels + the partially covered rim
    assert xs.min() >= 39 and xs.max() <= 56 and ys.min() >= 23 and ys.max() <= 40


def test_committed_fixture_matches_the_source_file(tmp_path):
    """The fixture is what the loader makes of paris-30k.svg. The source file (14 MB) is stood in
    for by tests/golden/paris30k_excerpt.npz (tests/golden/make_paris_excerpt.py): digests of its
    whole parse, and a seeded sample of its <path> elements, parsed afresh here."""
    gold = np.load(os.path.join(ROOT, "tests", "golden", "paris30k_excerpt.npz"))
    fixture = svg.PathList.load(os.path.join(ROOT, "tests", "data", "paris30k_paths.npz"))
    for k in ("cmd", "pts", "cmd_off", "pt_off", "color", "fill_rule"):
        a = getattr(fixture, k)
        got = hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + np.ascontiguousarray(a).tobytes()).hexdigest()
        assert got == str(gold["sha256_" + k]), k
    doc = tmp_path / "paris30k_excerpt.svg"
    doc.write_bytes(gold["svg"].tobytes())
    fresh = svg.parse_svg(str(doc))
    index = gold["index"]
    assert len(fresh) == len(index) > 300
    for j, i in enumerate(index):
        assert np.array_equal(fresh.cmd[fresh.cmd_off[j]:fresh.cmd_off[j + 1]], fixture.cmd[fixture.cmd_off[i]:fixture.cmd_off[i + 1]]), i
        assert np.array_equal(fresh.pts[fresh.pt_off[j]:fresh.pt_off[j + 1]], fixture.pts[fixture.pt_off[i]:fixture.pt_off[i + 1]]), i
        assert np.array_equal(fresh.color[j], fixture.color[i]) and fresh.fill_rule[j] == fixture.fill_rule[i], i
    assert len(fresh.weights) == 0 and not fresh.gradients


def test_cli_refuses_without_a_device(parsed, tmp_path):
    import subprocess
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _, path = parsed
    p = subprocess.run([sys.executable, "-m", "forma_b200.render", path, str(tmp_path / "o.ppm"), "--width", "64", "--height", "64"],
                       capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)
    assert not (tmp_path / "o.ppm").exists()
