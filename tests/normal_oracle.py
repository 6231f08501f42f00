"""Host statement of the oriented normals (include/ddn_b200.h, ddn_point_normals and the fused-normal forms).

Per-point normals in float64 from the definition: the camera-frame normal of the grid point's pixel rotated into the
world and normalised as ``oracle/restatement_masks.transform_normals`` states it, negated when it faces away from the
camera, (0, 0, 0) for a non-finite normal or a grid point without a point.  Fused normals exactly as the kernels sum
them: rint(n * 2^20) per point and component, 64-bit integer sums per voxel (the voxels of
``cpu_backend.partial_sums_numpy``), Σq / ‖Σq‖ in float64 rounded to float32."""

from __future__ import annotations

import numpy as np

from oracle.restatement_masks import transform_normals

import cpu_backend as CB

NORMAL_FIX = np.float32(1 << 20)
TIE = 1e-6  # |n_c . r| / (|n_c| |r|) at or below this: the orientation may go either way


def view_normals(normal_map, cam_from_world, intr, votes, stride: int):
    """One view: normal_map [H,W,3], cam_from_world [3,4], intr (fx, fy, cx, cy), votes [Hs,Ws] u8 of the strided grid.
    Returns (normals [Hs,Ws,3] f64, tie [Hs,Ws] bool)."""
    normal_map = np.asarray(normal_map, np.float32)
    fx, fy, cx, cy = (float(v) for v in intr)
    nc = normal_map[::stride, ::stride].astype(np.float64)
    hs, ws = nc.shape[:2]
    assert votes.shape == (hs, ws)
    with np.errstate(invalid="ignore", over="ignore"):
        n = transform_normals(nc, cam_from_world, np.ones((hs, ws), bool)).reshape(hs, ws, 3)
    ys, xs = np.meshgrid(np.arange(hs) * stride, np.arange(ws) * stride, indexing="ij")
    ray = np.stack([(xs - cx) / fx, (ys - cy) / fy, np.ones_like(xs, dtype=np.float64)], -1)
    dot = (nc * ray).sum(-1)
    with np.errstate(invalid="ignore"):
        tie = np.abs(dot) <= TIE * np.linalg.norm(nc, axis=-1) * np.linalg.norm(ray, axis=-1)
    n = np.where((dot > 0)[..., None], -n, n)
    bad = ~np.isfinite(n).all(-1) | (votes == 255)
    n[bad] = 0.0
    return n, tie & ~bad


def point_normals(normal_maps, poses, intr, votes, stride: int):
    """All views: per-view lists (or stacked arrays) of maps and strided vote grids.  Returns (normals, tie) as lists of
    per-view [Hs_v,Ws_v,3] / [Hs_v,Ws_v] arrays."""
    out = [view_normals(normal_maps[v], poses[v], intr[v], votes[v], stride) for v in range(len(votes))]
    return [o[0] for o in out], [o[1] for o in out]


def quantize(normals32):
    """q = rint(n * 2^20) per component (float32 product, exact; round half to even)."""
    return np.rint(np.asarray(normals32, np.float32) * NORMAL_FIX).astype(np.int64)


def fused_normal_sums(xyz32, normals32, voxel, origin):
    """Per-voxel sums of the quantised normals of the given (participating) points, keys ascending; the voxels are
    those of cpu_backend.partial_sums_numpy.  Returns (keys, sums [M,3] i64)."""
    xyz32 = np.asarray(xyz32, np.float32).reshape(-1, 3)
    if len(xyz32) == 0:
        return np.zeros(0, np.int64), np.zeros((0, 3), np.int64)
    uk = CB.partial_sums_numpy(xyz32, np.zeros((len(xyz32), 3), np.uint8), voxel, origin)[0]
    _, keys = CB.canonical_keys(xyz32, voxel, origin)
    inv = np.searchsorted(uk, keys)
    sums = np.zeros((len(uk), 3), np.int64)
    np.add.at(sums, inv, quantize(normals32))
    return uk, sums


def final_normals(sums):
    """Σq / ‖Σq‖ in float64, rounded to float32; (0, 0, 0) where Σq = 0.  The norm is sqrt((x² + y²) + z²), in that
    order, as the kernels evaluate it."""
    s = np.asarray(sums, np.int64).astype(np.float64)
    norm = np.sqrt((s[:, 0] * s[:, 0] + s[:, 1] * s[:, 1]) + s[:, 2] * s[:, 2])
    out = np.zeros_like(s)
    nz = norm > 0
    out[nz] = s[nz] / norm[nz, None]
    return out.astype(np.float32)
