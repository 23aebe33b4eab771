"""CPU: every reference citation (file:line) in the header, the docs and the product docstrings points at an
existing line of the reference tree, whose line counts tests/golden/make_reference_golden.py stored in
tests/golden/reference_line_counts.json (file name -> lines of the longest file of that name)."""
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# e.g. tf_ops/tf_sampling.cu:111-176, tf_grouping.cpp:80-87, pointnet_util.py:18-60, model.py:22
CITE = re.compile(r"\b((?:[\w./]+/)?(?:tf_\w+|pointnet_util|tf_util|model|train|predict|semantic_dataset|"
                  r"test_tf_ops|test_interpolate|interpolate|kitti_predict)\.(?:cu|cpp|py)):(\d+)(?:-(\d+))?")


def test_reference_citations_resolve():
    with open(os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")) as f:
        lengths = json.load(f)
    sources = [os.path.join(ROOT, "include", "pn2_b200.h"), os.path.join(ROOT, "DESIGN.md"),
               os.path.join(ROOT, "INTEGRATION.md")]
    sources += glob.glob(os.path.join(ROOT, "open3d-pointnet2-semantic3d_b200", "**", "*.py"), recursive=True)
    sources += glob.glob(os.path.join(ROOT, "open3d-pointnet2-semantic3d_b200", "csrc", "*.cu*"))
    sources += [os.path.join(ROOT, "oracle", f) for f in ("pn2_oracle.c", "layers_ref.py", "ref_shim.cu")]
    bad, checked = [], 0
    for src in sources:
        for m in CITE.finditer(open(src, errors="replace").read()):
            name, lo, hi = os.path.basename(m.group(1)), int(m.group(2)), int(m.group(3) or m.group(2))
            n = lengths.get(name)
            if n is None:
                bad.append("%s cites %s: no such file in the reference" % (os.path.relpath(src, ROOT), m.group(0)))
                continue
            checked += 1
            if not (1 <= lo <= hi <= n):
                bad.append("%s cites %s but %s has %d lines" % (os.path.relpath(src, ROOT), m.group(0), name, n))
    assert checked > 100, checked
    assert not bad, "\n".join(bad[:20])
