"""Writes the stand-ins for the reference's files that tests compare with, so that the suite needs nothing outside the
repository:

  tests/golden/out.ppm.gz           the reference's engine/out.ppm: the oracle's demo render (800x600), checked to have
                                    the sha256 recorded from the reference's file in out_ppm.json
  tests/golden/cornell_box.obj      the geometry of the reference's test_data/*.obj, written back from the meshes parsed
  tests/golden/dodecahedron.obj     out of those files (rusty_marcher_b200/scenes/*.npz): one object per model, its
                                    triangles in the order the reader produced them, no materials (the engine ignores them)

    python tests/golden/make_reference_inputs.py
"""
import gzip
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import oracle as O  # noqa: E402
from rusty_marcher_b200 import workloads  # noqa: E402


def write_obj(name):
    verts, index, lines = [], {}, []
    for model, tris in workloads.load_models(name):
        lines.append("o %s" % model)
        for tri in tris:
            for v in map(tuple, tri):
                if v not in index:
                    index[v] = len(index) + 1
                    verts.append("v " + " ".join(np.format_float_positional(np.float32(c), trim="-") for c in v))
            lines.append("f " + " ".join(str(index[v]) for v in map(tuple, tri)))
    with open(os.path.join(GOLDEN, name + ".obj"), "w") as f:
        f.write("\n".join(verts + lines) + "\n")


def main():
    meta = json.load(open(os.path.join(GOLDEN, "out_ppm.json")))
    rgb = O.render(O.Scene.create_default(), 800, 600)["rgb"]
    O.normalize(rgb)
    ppm = O.ppm_bytes(rgb)
    assert hashlib.sha256(ppm).hexdigest() == meta["sha256"], "the oracle no longer renders the reference's out.ppm"
    with open(os.path.join(GOLDEN, "out.ppm.gz"), "wb") as f:
        f.write(gzip.compress(ppm, 9, mtime=0))
    for name in ("cornell_box", "dodecahedron"):
        write_obj(name)
        s = O.Scene()
        s.add_obj_file(os.path.join(GOLDEN, name + ".obj"), offset=(0., 0., 0.))
        models = workloads.load_models(name)
        assert s.num_shapes == len(models) and all(np.array_equal(s.obj_triangles(i), v) for i, (_n, v) in enumerate(models))


if __name__ == "__main__":
    main()
