"""Fixture generator (needs a checkout of the reference and oracle/_ref/libbxref.so, built from it by
oracle/ref_build/build_ref.py): what two groups of tests compare against, so that they run without the reference.
  tests/golden/reference_layout.json  every Python file of the reference checkout, by relative path (names only, no code):
                                      the tree test_dropin.py rebuilds to check how the documented PYTHONPATH resolves
  tests/golden/reference_cpp.json     shape + hash of what the reference's own neighbors.cpp / grid_subsampling.cpp return on
                                      the inputs of the a17 / a18 tests of test_oracle_cpu.py
    python tests/tools/gen_reference_golden.py REFERENCE_CHECKOUT"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import oracle as O  # noqa: E402
import test_oracle_cpu as T  # noqa: E402

ref_root = os.path.realpath(sys.argv[1])
layout = []
for d, dirs, files in os.walk(ref_root):
    dirs[:] = sorted(x for x in dirs if not x.startswith("."))
    layout += [os.path.relpath(os.path.join(d, f), ref_root) for f in sorted(files) if f.endswith(".py")]
assert "utils/timer.py" in layout and "models/BUFFERX.py" in layout, "not a checkout of the reference"

if not O.ref_available():
    sys.exit("oracle/_ref/libbxref.so is missing: build it with oracle/ref_build/build_ref.py")
cpp = {"radius_neighbors": {}, "grid_subsampling": {}}
for radius, qb, sb in T.RADIUS_CASES:
    q, s = T.radius_inputs(radius, qb, sb)
    b = O.ref_radius_neighbors(q, s, qb, sb, radius)
    cpp["radius_neighbors"][str(radius)] = {"shape": list(b.shape), "sha": T.sha(b)}
pts = T.grid_points()
for dl in T.GRID_DLS:
    b = T.sorted_rows(O.ref_grid_subsampling(pts, dl))
    cpp["grid_subsampling"][str(dl)] = {"shape": list(b.shape), "sha": T.sha(b)}

for name, obj in (("reference_layout.json", layout), ("reference_cpp.json", cpp)):
    p = os.path.join(ROOT, "tests", "golden", name)
    with open(p, "w") as f:
        json.dump(obj, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", p, os.path.getsize(p), "bytes")
