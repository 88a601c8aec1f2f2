"""The marching-cubes case table (isaac_ros_nvblox_b200/csrc/nvb_mc_table.h and the oracle's copy oracle/mc_table.h):
the two copies are equal, the table satisfies the invariants of the published table (every triangle uses only edges whose two
corners lie on opposite sides of the surface; complementary configurations have the same edges), and every row equals the
reference's (nvblox/include/nvblox/mesh/internal/impl/marching_cubes_table.h:34-333), stored as
tests/golden/reference_mc_table.npz by tests/golden/make_reference_mc_table.py."""
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "tests", "golden", "reference_mc_table.npz")
EDGE_CORNERS = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]


def _rows(path):
    src = open(path).read()
    body = src[src.index("kMcTriangles[256]"):]
    body = body[body.index("{") + 1:body.index("};")]
    rows = re.findall(r'"([0-9a-b]*)"', body)
    assert len(rows) == 256
    return [[int(c, 16) for c in r] for r in rows]


def test_product_and_oracle_tables_are_equal():
    assert _rows(os.path.join(ROOT, "isaac_ros_nvblox_b200", "csrc", "nvb_mc_table.h")) == _rows(os.path.join(ROOT, "oracle", "mc_table.h"))


def test_table_invariants():
    rows = _rows(os.path.join(ROOT, "oracle", "mc_table.h"))
    assert rows[0] == [] and rows[255] == []
    for cfg, row in enumerate(rows):
        assert len(row) % 3 == 0 and len(row) <= 15
        crossing = {e for e, (a, b) in enumerate(EDGE_CORNERS) if ((cfg >> a) & 1) != ((cfg >> b) & 1)}
        assert set(row) == crossing, cfg  # every crossing edge carries a vertex, no other edge does
        for t in range(0, len(row), 3):
            assert len(set(row[t:t + 3])) == 3
        assert set(rows[255 - cfg]) == crossing
    assert sum(len(r) // 3 for r in rows) == 820  # triangles in the published table


def test_table_equals_the_reference_table():
    g = np.load(REF)
    ref, nt = g["triangle_table"].tolist(), g["num_triangles"].tolist()
    assert len(ref) == 256
    rows = _rows(os.path.join(ROOT, "oracle", "mc_table.h"))
    for cfg in range(256):
        assert [v for v in ref[cfg] if v >= 0] == rows[cfg], cfg
    assert [len(r) // 3 for r in rows] == nt
