"""On-disk formats (SURVEY 8f rank 3): PCD / KITTI .bin readers into the ABI's AoS48 layout, pose writer."""
import hashlib
import os

import numpy as np
import pytest

from mulls_b200 import io as mio

DEMO_PCD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "demo_000000_head.pcd")
DEMO_PCD_ROWS_SHA256 = "a86107f2ea8e9b8885df7e1df072a91d6061519b70d139259ef3c772691af73b"


def _write_pcd(path, arr, fields, binary=True):
    with open(path, "wb") as f:
        hdr = ("# .PCD v0.7 - Point Cloud Data file format\nVERSION 0.7\nFIELDS %s\nSIZE %s\nTYPE %s\nCOUNT %s\n"
               "WIDTH %d\nHEIGHT 1\nVIEWPOINT 0 0 0 1 0 0 0\nPOINTS %d\nDATA %s\n") % (
            " ".join(fields), " ".join(["4"] * len(fields)), " ".join(["F"] * len(fields)),
            " ".join(["1"] * len(fields)), len(arr), len(arr), "binary" if binary else "ascii")
        f.write(hdr.encode())
        if binary:
            f.write(arr.astype("<f4").tobytes())
        else:
            for row in arr:
                f.write((" ".join(repr(float(v)) for v in row) + "\n").encode())


@pytest.mark.parametrize("binary", [True, False])
def test_read_pcd_roundtrip(tmp_path, binary):
    rng = np.random.default_rng(0)
    fields = ["x", "y", "z", "intensity", "normal_x", "normal_y", "normal_z", "curvature"]
    arr = rng.normal(size=(257, 8)).astype(np.float32)
    p = str(tmp_path / "a.pcd")
    _write_pcd(p, arr, fields, binary)
    c = mio.read_pcd(p)
    assert c.shape == (257, 12) and c.flags["C_CONTIGUOUS"] and c.dtype == np.float32
    np.testing.assert_array_equal(c[:, [0, 1, 2, 8, 4, 5, 6, 9]], arr)
    assert (c[:, 3] == 1.0).all() and (c[:, [7, 10, 11]] == 0).all()
    # xyz-only file
    _write_pcd(p, arr[:, :3], ["x", "y", "z"], binary)
    c = mio.read_pcd(p)
    np.testing.assert_array_equal(c[:, 0:3], arr[:, :3])
    assert (c[:, 4:10] == 0).all()


def test_read_kitti_bin_and_block(tmp_path):
    rng = np.random.default_rng(1)
    raw = rng.uniform(-50, 50, size=(100, 4)).astype(np.float32)
    raw[:, 3] = rng.uniform(0, 1, 100)
    p = str(tmp_path / "000000.bin")
    raw.tofile(p)
    c = mio.read_kitti_bin(p)
    assert c.shape == (101, 12)                      # the reference's read loop appends one default point
    np.testing.assert_array_equal(c[:100, 0:3], raw[:, 0:3])
    np.testing.assert_array_equal(c[:100, 8], raw[:, 3] * np.float32(255))
    assert (c[100, [0, 1, 2, 8]] == 0).all()
    assert mio.read_kitti_bin(p, reference_eof_point=False).shape == (100, 12)
    blk = mio.read_cloud_block(p, normalize_intensity=True)
    assert abs(blk["pc_raw"][:, 8].max() - 255.0) < 1e-3 and blk["pc_raw"][:, 8].min() == 0.0
    b = blk["local_bound"]
    assert b[0] <= raw[:, 0].min() and b[3] >= raw[:, 0].max()


def test_pose_writer(tmp_path):
    T = np.eye(4)
    T[:3, 3] = (1.23456789012, -2.5, 1e-9)
    p = str(tmp_path / "pose.txt")
    mio.write_lo_pose_overwrite(T, p)
    mio.write_lo_pose_append(T, p)
    lines = open(p).read().splitlines()
    assert len(lines) == 2 and lines[0] == lines[1]
    vals = [float(v) for v in lines[0].split()]
    assert len(vals) == 12 and vals[3] == 1.2345679 and vals[7] == -2.5 and vals[11] == 1e-9


def test_reads_reference_demo_scan():
    """The first 4096 points of MULLS's demo scan 000000 (tests/golden/make_golden_pcd.py): the rows must be what the
    reader made of the original 124 668-point file."""
    c = mio.read_pcd(DEMO_PCD)
    assert c.shape == (4096, 12)
    assert abs(np.linalg.norm(c[:1000, 4:7], axis=1) - 1.0).max() < 1e-3
    assert hashlib.sha256(c.tobytes()).hexdigest() == DEMO_PCD_ROWS_SHA256


# ---- the native readers of the C-ABI (csrc/scan_io.h) against the numpy ones above: bit for bit -------------------

@pytest.mark.parametrize("binary", [True, False])
def test_native_pcd_reader_equals_the_numpy_one(tmp_path, binary):
    rng = np.random.default_rng(3)
    fields = ["x", "y", "z", "intensity", "normal_x", "normal_y", "normal_z", "curvature"]
    arr = rng.normal(size=(1031, 8)).astype(np.float32)
    arr[:, 3] = rng.uniform(0, 200, 1031)
    p = str(tmp_path / "b.pcd")
    for cols, names in ((slice(0, 8), fields), (slice(0, 3), fields[:3]), (slice(0, 4), ["x", "y", "z", "rgb"])):
        _write_pcd(p, arr[:, cols], names, binary)
        for norm in ((False, True) if "intensity" in names else (False,)):  # (constant intensity: 255 / 0 in the reference too)
            a = mio.read_cloud_block(p, normalize_intensity=norm)
            b = mio.read_cloud_block_native(p, normalize_intensity=norm)
            assert b["pc_raw"].shape == a["pc_raw"].shape
            np.testing.assert_array_equal(b["pc_raw"].view(np.uint32), a["pc_raw"].view(np.uint32))
            assert b["local_bound"] == tuple(a["local_bound"])


def test_native_kitti_reader_equals_the_numpy_one(tmp_path):
    rng = np.random.default_rng(4)
    raw = rng.uniform(-50, 50, size=(777, 4)).astype(np.float32)
    raw[:, 3] = rng.uniform(0, 1, 777)
    p = str(tmp_path / "000123.bin")
    raw.tofile(p)
    for norm in (False, True):
        a = mio.read_cloud_block(p, normalize_intensity=norm)
        b = mio.read_cloud_block_native(p, normalize_intensity=norm)
        assert b["pc_raw"].shape == (778, 12)  # the reference's end-of-file point
        np.testing.assert_array_equal(b["pc_raw"].view(np.uint32), a["pc_raw"].view(np.uint32))
        assert b["local_bound"] == tuple(a["local_bound"])


def test_native_reader_errors_and_pose_writer(tmp_path):
    import ctypes as C

    from mulls_b200 import abi

    lib = abi.load_library()
    n = C.c_size_t(0)
    assert lib.mulls_scan_probe(str(tmp_path / "missing.pcd").encode(), C.byref(n)) == -105  # MULLS_E_IO
    p = str(tmp_path / "c.pcd")
    _write_pcd(p, np.zeros((10, 3), np.float32), ["x", "y", "z"], True)
    rows = np.empty((4, 12), np.float32)
    assert lib.mulls_scan_read(p.encode(), rows.ctypes.data_as(C.POINTER(C.c_float)), 4, C.byref(n), None, 0) == -102  # capacity
    blob = open(p, "rb").read().replace(b"DATA binary", b"DATA binary_compressed")
    open(p, "wb").write(blob)
    assert lib.mulls_scan_probe(p.encode(), C.byref(n)) == -103  # MULLS_E_UNSUPPORTED
    T = np.eye(4)
    T[:3, 3] = (1.23456789012, -2.5, 1e-9)
    T[0, 1] = 0.333333333333
    a, b = str(tmp_path / "a.txt"), str(tmp_path / "b.txt")
    mio.write_lo_pose_overwrite(T, a), mio.write_lo_pose_append(T, a)
    assert mio.write_lo_pose_native(T, b, overwrite=True) and mio.write_lo_pose_native(T, b)
    assert open(a).read() == open(b).read()


def test_native_reader_on_the_reference_demo_scan():
    a = mio.read_pcd(DEMO_PCD)
    b = mio.read_cloud_block_native(DEMO_PCD)
    np.testing.assert_array_equal(b["pc_raw"].view(np.uint32), a.view(np.uint32))
