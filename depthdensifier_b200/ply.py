"""Oriented point clouds as binary PLY: the vertex layout of COLMAP's ``fused.ply`` and of 3D Gaussian Splatting's
``storePly`` / ``fetchPly`` (``float x y z nx ny nz``, ``uchar red green blue``; 27 bytes per vertex, little endian)."""

from __future__ import annotations

from pathlib import Path

import numpy as np

VERTEX_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4"),
                         ("red", "u1"), ("green", "u1"), ("blue", "u1")])


def ply_header(n: int) -> bytes:
    props = "".join(f"property {'float' if VERTEX_DTYPE[name].kind == 'f' else 'uchar'} {name}\n" for name in VERTEX_DTYPE.names)
    return f"ply\nformat binary_little_endian 1.0\nelement vertex {int(n)}\n{props}end_header\n".encode("ascii")


def write_ply(path, xyz, normals, rgb) -> None:
    """Writes ``xyz`` [N,3] (as float32), ``normals`` [N,3] (as float32) and ``rgb`` [N,3] u8 to ``path``."""
    xyz = np.asarray(xyz).reshape(-1, 3)
    normals = np.asarray(normals).reshape(-1, 3)
    rgb = np.asarray(rgb).reshape(-1, 3)
    n = len(xyz)
    if len(normals) != n or len(rgb) != n:
        raise ValueError(f"xyz, normals and rgb differ in length: {n}, {len(normals)}, {len(rgb)}")
    if rgb.dtype != np.uint8:
        raise ValueError(f"rgb must be uint8, got {rgb.dtype}")
    v = np.empty(n, VERTEX_DTYPE)
    v["x"], v["y"], v["z"] = xyz.astype(np.float32).T
    v["nx"], v["ny"], v["nz"] = normals.astype(np.float32).T
    v["red"], v["green"], v["blue"] = rgb.T
    with open(Path(path), "wb") as f:
        f.write(ply_header(n))
        f.write(v.tobytes())
