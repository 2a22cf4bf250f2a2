"""Stores what paris-30k.svg parses to, small enough to commit, for
tests/test_svg_loader.py::test_committed_fixture_matches_the_source_file.

    python tests/golden/make_paris_excerpt.py <path to forma's assets/svgs/paris-30k.svg>

The source file is 14 MB; the test needs it to check that tests/data/paris30k_paths.npz is
what forma_b200/svg.py makes of it. The output tests/golden/paris30k_excerpt.npz keeps:
  svg           a valid SVG document (uint8 UTF-8 bytes): the file with every <path> element
                outside a seeded sample removed; its groups and the sampled paths are verbatim
  index         int64: the position of every sampled <path> in the file (= its fixture path)
  sha256_<key>  digest of every array of the whole file's parse (dtype, shape and bytes)
"""
import hashlib
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from forma_b200 import svg  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "paris30k_excerpt.npz")
KEYS = ("cmd", "pts", "cmd_off", "pt_off", "color", "fill_rule")
BUDGET = 96 << 10  # bytes of sampled <path> elements


def digest(a):
    return hashlib.sha256(a.dtype.str.encode() + str(a.shape).encode() + np.ascontiguousarray(a).tobytes()).hexdigest()


def main(src):
    text = open(src, encoding="utf-8").read()
    elems = list(re.finditer(r"<path\b[^>]*/>", text))
    full = svg.parse_svg(src)
    assert len(elems) == len(full), (len(elems), len(full))
    rng = np.random.default_rng(2160)
    picked, size = [], 0
    for i in rng.permutation(len(elems)):
        n = elems[i].end() - elems[i].start()
        if size + n <= BUDGET:
            picked.append(int(i))
            size += n
    picked.sort()
    keep, doc, end = set(picked), [text[:elems[0].start()]], elems[0].start()
    for i, e in enumerate(elems):
        gap = text[end:e.start()]
        if gap.strip():  # <g> tags and their attributes stay; whitespace between elements goes
            doc.append(gap)
        if i in keep:
            doc.append(e.group(0))
        end = e.end()
    doc = "".join(doc) + text[end:]
    arrays = {"svg": np.frombuffer(doc.encode("utf-8"), np.uint8), "index": np.array(picked, np.int64)}
    arrays.update({"sha256_" + k: np.array(digest(getattr(full, k))) for k in KEYS})
    np.savez_compressed(OUT, **arrays)
    print(f"{len(picked)} of {len(elems)} paths, {len(doc)} bytes of SVG -> {OUT} ({os.path.getsize(OUT)} bytes)")


if __name__ == "__main__":
    main(sys.argv[1])
