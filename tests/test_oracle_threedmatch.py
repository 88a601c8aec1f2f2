"""The oracle on REFERENCE-HELD real data: the five 3DMatch frames the reference ships for its own tests
(nvblox/tests/data/3dmatch/seq-01, real 640x480 16-bit depth with ~13 % invalid pixels, poses, intrinsics, one colour image),
stored raw in tests/golden/threedmatch_seq01.npz by tests/golden/make_threedmatch_fixture.py.
  * the fixture's inputs are the reference's files, bit for bit: their SHA-256, taken from the reference's files when the
    fixture was made, is stored in tests/golden/threedmatch_seq01_sources.json;
  * the reference's own loader known answers (tests/test_3dmatch.cpp:60-87) hold for the fixture;
  * the oracle reproduces the committed per-frame block lists and layer checksums (TSDF + colour + ESDF).
The CUDA path is compared with the oracle on the same frames in tests/test_gpu_bench_pipeline.py."""
import json
import os
import sys

import numpy as np
import pytest

from helpers import ESDF_FIELDS, layer_checksum

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import make_threedmatch_fixture as mk  # noqa: E402


@pytest.fixture(scope="module")
def fx():
    return np.load(os.path.join(GOLDEN, "threedmatch_seq01.npz"))


def test_fixture_inputs_are_the_reference_files(fx):
    with open(mk.SOURCES) as f:
        want = json.load(f)
    assert mk.input_digests(*(fx[k] for k in mk.INPUTS)) == want


def test_reference_loader_known_answers(fx):
    mk.check_loader_kats(fx["intrinsics"], fx["depth_u16"])
    d = mk.depth_to_float(fx["depth_u16"])
    assert d.dtype == np.float32 and d.shape == (5, 480, 640)
    assert 0.05 < float((fx["depth_u16"][0] == 0).mean()) < 0.25  # real sensor data: invalid pixels are zeros
    for T in fx["poses"]:  # poses are rigid (Fuser checks det(R) ~ 1, executables/src/datasets/3dmatch.cpp:252)
        assert abs(np.linalg.det(T[:3, :3].astype(np.float64)) - 1.0) < 1e-4 and np.array_equal(T[3], [0, 0, 0, 1])


def test_oracle_reproduces_the_committed_results(fx):
    o, lists = mk.run_oracle(fx["intrinsics"], fx["depth_u16"], fx["poses"], fx["color0"], float(fx["voxel_size"]))
    for i, b in enumerate(lists):
        assert np.array_equal(b, fx["blocks_%d" % i]), i
    assert len(o.tsdf_layer()) == int(fx["num_tsdf_blocks"])
    assert layer_checksum(o.tsdf_layer(), ("distance", "weight")) == int(fx["tsdf_checksum"])
    assert layer_checksum(o.esdf_layer(), ESDF_FIELDS) == int(fx["esdf_checksum"])
    assert layer_checksum(o.color_layer(), ("color", "weight")) == int(fx["color_checksum"])
    # real data exercises what the synthetic scenes do not: invalid (zero) depth, unobserved voxels inside allocated blocks
    esdf = o.esdf_layer()
    obs = np.concatenate([b["observed"].ravel() for b in esdf.values()]).astype(bool)
    site = np.concatenate([b["is_site"].ravel() for b in esdf.values()]).astype(bool)
    assert 0.2 < obs.mean() < 0.95 and site.sum() > 5000 and not (site & ~obs).any()
