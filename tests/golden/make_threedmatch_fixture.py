"""Builds tests/golden/threedmatch_seq01.npz from the reference's own test data
(nvblox/tests/data/3dmatch: five 640x480 16-bit depth PNGs of seq-01 with poses, camera-intrinsics.txt, the colour image of
frame 0) and the oracle's results on them, and tests/golden/threedmatch_seq01_sources.json: the SHA-256 of every input
array as read from the reference's files, which tests/test_oracle_threedmatch.py checks the fixture against. Run with the root
of an isaac_ros_nvblox checkout:

    python tests/golden/make_threedmatch_fixture.py <isaac_ros_nvblox checkout>

The inputs are stored raw (uint16 millimetres, float32 poses parsed like parsePoseFromFile /
parseCameraFromFile, nvblox/executables/src/datasets/3dmatch.cpp:31-75) so that the tests run the same frames without the
reference tree; the depth conversion is io::readFromPng's (nvblox/src/io/image_io.cpp:117-154):
float(u16) * kDefaultUintDepthScaleFactor, kDefaultUintDepthScaleFactor = 1.0f / 1000.0f (nvblox/include/nvblox/io/image_io.h:32).
The loader known answers of nvblox/tests/test_3dmatch.cpp:60-87 are asserted here and in tests/test_oracle_threedmatch.py.
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
DATA = os.path.join("nvblox_ros", "nvblox_core", "nvblox", "tests", "data", "3dmatch")
FRAMES = (0, 1, 2, 116, 422)
OUT = os.path.join(ROOT, "tests", "golden", "threedmatch_seq01.npz")
SOURCES = os.path.join(ROOT, "tests", "golden", "threedmatch_seq01_sources.json")
INPUTS = ("intrinsics", "depth_u16", "poses", "color0")
VOXEL = 0.05


def load_reference_data(checkout):
    from PIL import Image
    data = os.path.join(checkout, DATA)
    K = np.array([[np.float32(t) for t in line.split()] for line in open(os.path.join(data, "camera-intrinsics.txt")) if line.strip()],
                 np.float32)
    depth, poses = [], []
    for f in FRAMES:
        base = os.path.join(data, "seq-01", "frame-%06d" % f)
        d = np.array(Image.open(base + ".depth.png"))
        assert d.dtype == np.uint16 and d.shape == (480, 640)
        depth.append(d)
        poses.append(np.array([[np.float32(t) for t in line.split()] for line in open(base + ".pose.txt") if line.strip()], np.float32))
    color0 = np.array(Image.open(os.path.join(data, "seq-01", "frame-000000.color.png")).convert("RGB"), np.uint8)
    assert color0.shape == (480, 640, 3)
    return K, np.stack(depth), np.stack(poses), color0


def input_digests(*arrays):
    """{input name: "dtype shape sha256"} of the arrays INPUTS names, in that order."""
    return {k: "%s %s %s" % (a.dtype.str, "x".join(map(str, a.shape)), hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest())
            for k, a in zip(INPUTS, arrays)}


def depth_to_float(depth_u16):
    """io::readFromPng: static_cast<float>(u16) * (1.0f / 1000.0f), one binary32 multiplication."""
    return depth_u16.astype(np.float32) * (np.float32(1.0) / np.float32(1000.0))


def check_loader_kats(K, depth_u16):
    """Dataset3DMatchTest.ParseCameraFromFile / LoadImage (nvblox/tests/test_3dmatch.cpp:60-87)."""
    K_true = np.array([[5.70342205e+02, 0, 3.2e+02], [0, 5.70342205e+02, 2.4e+02], [0, 0, 1]], np.float32)
    assert np.allclose(K, K_true, rtol=1e-5)
    d = depth_to_float(depth_u16[0])
    assert d.shape == (480, 640) and abs(float(d.min()) - 0.0) < 1e-4 and abs(float(d.max()) - 7.835) < 1e-4


def run_oracle(K, depth_u16, poses, color0, voxel=VOXEL):
    """Depth frames in file order, the colour image after the first depth frame, an ESDF update after every frame."""
    from oracle import oracle as orc
    cam = orc.Camera(float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]), 640, 480)
    o = orc.OracleMap(voxel)
    lists = []
    for i in range(len(depth_u16)):
        b = o.integrate_depth(depth_to_float(depth_u16[i]), poses[i], cam)
        if i == 0:
            o.integrate_color(color0, poses[0], cam)
        o.integrate_esdf(b)
        lists.append(b)
    return o, lists


def main():
    from helpers import ESDF_FIELDS, layer_checksum
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    K, depth, poses, color0 = load_reference_data(sys.argv[1])
    check_loader_kats(K, depth)
    o, lists = run_oracle(K, depth, poses, color0)
    out = dict(intrinsics=K, depth_u16=depth, poses=poses, color0=color0, frames=np.array(FRAMES), voxel_size=np.float32(VOXEL),
               tsdf_checksum=np.int64(layer_checksum(o.tsdf_layer(), ("distance", "weight"))),
               esdf_checksum=np.int64(layer_checksum(o.esdf_layer(), ESDF_FIELDS)),
               color_checksum=np.int64(layer_checksum(o.color_layer(), ("color", "weight"))),
               num_tsdf_blocks=np.int64(len(o.tsdf_layer())))
    for i, b in enumerate(lists):
        out["blocks_%d" % i] = b
    np.savez_compressed(OUT, **out)
    with open(SOURCES, "w") as f:
        json.dump(input_digests(K, depth, poses, color0), f, indent=1)
        f.write("\n")
    print("wrote", OUT, os.path.getsize(OUT), "bytes;", len(o.tsdf_layer()), "tsdf blocks; lists", [len(b) for b in lists])


if __name__ == "__main__":
    main()
