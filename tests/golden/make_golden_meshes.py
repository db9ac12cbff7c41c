"""The reference's two example meshes (examples/wand.obj, examples/screwdriver.obj: the README's `--mc` example), read with
mesh_to_pc.SimpleMesh.load_obj and stored as tests/golden/example_meshes.npz: <name>_vertices fp32 [V, 3],
<name>_faces int32 [F, 3].  The wand has two faces whose three indices are equal (zero-area triangles).
Used by tests/test_watertight.py and tools/bench_watertight.py.

usage: python tests/golden/make_golden_meshes.py <reference checkout>
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from mesh_to_pc import SimpleMesh  # noqa: E402

NAMES = ("wand", "screwdriver")


def main(ref):
    arrays = {}
    for name in NAMES:
        m = SimpleMesh.load_obj(os.path.join(ref, "examples", name + ".obj"))
        arrays[name + "_vertices"] = m.vertices.astype(np.float32)
        arrays[name + "_faces"] = m.faces.astype(np.int32)
        print(name, m.vertices.shape, m.faces.shape)
    out = os.path.join(HERE, "example_meshes.npz")
    np.savez_compressed(out, **arrays)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
