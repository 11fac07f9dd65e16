"""Re-encode the reference's only data asset, meshes/original.obj (canonical body mesh of frame 0,
meshes/README:1), as a compact npz fixture for tests and benchmarks.

Needs a reference checkout (oracle/_ref/ or $DFB_REFERENCE_ROOT):  python tests/golden/make_mesh_fixture.py
OBJ parsing follows the reference's own loader semantics (core/meshutil.py:12-39: 'v' lines -> vertices,
'f' lines -> first index of each a/b/c triple, 0-based if the minimum index is 0).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("DFB_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle", "_ref"))
OUT = os.path.join(HERE, "body_mesh.npz")


def main():
    v, n, f = [], [], []
    for line in open(os.path.join(REF, "meshes", "original.obj")):
        t = line.split()
        if not t:
            continue
        if t[0] == "v":
            v.append(t[1:4])
        elif t[0] == "vn":
            n.append(t[1:4])
        elif t[0] == "f":
            f.append([int(x.split("/")[0]) for x in t[1:4]])
    v = np.array(v, dtype=np.float32)
    n = np.array(n, dtype=np.float32)
    f = np.array(f, dtype=np.int32)
    if f.min() == 1:
        f -= 1
    np.savez_compressed(OUT, vertices=v, normals=n, faces=f)
    print("wrote", OUT, v.shape, n.shape, f.shape, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    sys.exit(main())
