"""write_ply: the bytes of the binary PLY against a hand-built header and struct layout, a round trip through a reader of
the format, and an empty cloud."""

import struct

import numpy as np
import pytest

from depthdensifier_b200.ply import write_ply

HEADER = (b"ply\nformat binary_little_endian 1.0\nelement vertex %d\n"
          b"property float x\nproperty float y\nproperty float z\n"
          b"property float nx\nproperty float ny\nproperty float nz\n"
          b"property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")


def read_ply(path):
    """A reader of the binary little-endian PLYs 3DGS's fetchPly takes: (xyz, normals, rgb)."""
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    assert lines[0] == "ply" and lines[1] == "format binary_little_endian 1.0"
    n = int(next(ln for ln in lines if ln.startswith("element vertex")).split()[-1])
    props = [ln.split() for ln in lines if ln.startswith("property")]
    dt = np.dtype([(name, "<f4" if kind == "float" else "u1") for _, kind, name in props])
    v = np.frombuffer(data[end:], dt, count=n)
    assert len(data) == end + n * dt.itemsize
    return (np.stack([v["x"], v["y"], v["z"]], 1), np.stack([v["nx"], v["ny"], v["nz"]], 1),
            np.stack([v["red"], v["green"], v["blue"]], 1))


def test_bytes(tmp_path):
    xyz = np.array([[1.0, -2.5, 3.25], [0.1, 0.2, 0.3]])
    nrm = np.array([[0.0, 0.0, 1.0], [0.6, -0.8, 0.0]], np.float32)
    rgb = np.array([[255, 0, 7], [1, 2, 3]], np.uint8)
    p = tmp_path / "a.ply"
    write_ply(p, xyz, nrm, rgb)
    want = HEADER % 2 + b"".join(struct.pack("<6f3B", *map(float, xyz[i]), *map(float, nrm[i]), *map(int, rgb[i])) for i in range(2))
    assert p.read_bytes() == want
    assert len(want) == len(HEADER % 2) + 2 * 27


def test_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    xyz = rng.normal(size=(1000, 3)).astype(np.float32)
    nrm = rng.normal(size=(1000, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, (1000, 3), dtype=np.uint8)
    write_ply(tmp_path / "b.ply", xyz, nrm, rgb)
    x, n, c = read_ply(tmp_path / "b.ply")
    assert np.array_equal(x, xyz) and np.array_equal(n, nrm) and np.array_equal(c, rgb)


def test_empty(tmp_path):
    write_ply(tmp_path / "e.ply", np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 3), np.uint8))
    assert (tmp_path / "e.ply").read_bytes() == HEADER % 0
    x, n, c = read_ply(tmp_path / "e.ply")
    assert x.shape == n.shape == c.shape == (0, 3)


def test_rejects_mismatched_inputs(tmp_path):
    with pytest.raises(ValueError):
        write_ply(tmp_path / "x.ply", np.zeros((2, 3)), np.zeros((1, 3)), np.zeros((2, 3), np.uint8))
    with pytest.raises(ValueError):
        write_ply(tmp_path / "x.ply", np.zeros((2, 3)), np.zeros((2, 3)), np.zeros((2, 3), np.int32))
