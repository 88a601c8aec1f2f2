"""Builds tests/golden/reference_mc_table.npz: the marching-cubes tables of the reference (kTriangleTable[256][16] and
kNumTrianglesTable[256] of nvblox/include/nvblox/mesh/internal/impl/marching_cubes_table.h:34-333) as plain arrays, so that
tests/test_mesh_table.py compares the project's table with them wherever it runs. Run with the root of an isaac_ros_nvblox
checkout:

    python tests/golden/make_reference_mc_table.py <isaac_ros_nvblox checkout>
"""
import os
import re
import sys

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_mc_table.npz")
TABLE = os.path.join("nvblox_ros", "nvblox_core", "nvblox", "include", "nvblox", "mesh", "internal", "impl", "marching_cubes_table.h")


def parse(path):
    """-> (triangle_table (256, 16) int8, -1 padded; num_triangles (256,) int32)."""
    src = open(path).read()
    body = src[src.index("kTriangleTable[256][16]"):]
    body = body[body.index("{") + 1:body.index("};")]
    tri = np.array([[int(x) for x in re.findall(r"-?\d+", r)] for r in re.findall(r"\{([^{}]*)\}", body)], np.int8)
    nt = src[src.index("kNumTrianglesTable[256]"):]
    nt = np.array([int(x) for x in re.findall(r"\d+", nt[nt.index("{"):nt.index("};")])], np.int32)
    assert tri.shape == (256, 16) and nt.shape == (256,)
    return tri, nt


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    tri, nt = parse(os.path.join(sys.argv[1], TABLE))
    np.savez_compressed(OUT, triangle_table=tri, num_triangles=nt)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
