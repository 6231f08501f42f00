"""TEST INFRASTRUCTURE ONLY - CPU restatement of the reference densification hot path.

This file is the parity oracle.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it; the product package
``depthdensifier_b200`` never does and fails loudly when its CUDA library is missing.

Parity status
-------------
* Rows A1-A7, B1-B4, C1-C5 (SURVEY.md §8a) restate /root/reference code and are PINNED:
  ``tests/test_oracle_vs_reference.py`` runs the reference's unmodified ``main()`` and
  ``DepthRefiner.refine_depth`` (via ``oracle/run_reference.py``) and asserts bit-identical points,
  colours, votes, keep masks and refined depth at K = V; ``tests/golden/*.npz`` holds the same
  outputs for machines without ``/root/reference``.
* Rows N1-N5 (affine alignment, bilinear/two-sided consistency, voxel fusion, sparse merge) have
  NO reference implementation: **parity unpinned** - they are defined here (SURVEY.md §8a-new).

Arithmetic follows the reference exactly: stage 1 in torch CPU float32 (the reference's own
library calls), stages 2-3 in numpy float64 on float32 maps.
"""

from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------
# Stage 1: per-view depth alignment (reference: src/depthdensifier/depth_refiner.py)
# --------------------------------------------------------------------------------------
@dataclass
class AlignConfig:
    """Mirror of RefinerConfig (depth_refiner.py:16-31) plus the north-star mode switch."""

    min_correspondences: int = 50
    edge_margin: int = 10
    robust: bool = True
    outlier_threshold: float = 2.5
    skip_smoothing: bool = False
    adaptive_correspondences: bool = True
    align_mode: str = "pwl"  # "pwl" = reference; "affine" = N1 (parity unpinned)
    max_pairs: int = 500  # depth_refiner.py:302-306


def project_sparse(points3D: torch.Tensor, cam_from_world: torch.Tensor, K: torch.Tensor):
    """A1 - depth_refiner.py:92-115.  float32; homogeneous 4x4 product, z>0 gate, 2x2 block of K."""
    n = points3D.shape[0]
    hom = torch.cat([points3D, torch.ones(n, 1, dtype=points3D.dtype)], dim=1)
    H4 = torch.cat([cam_from_world, torch.tensor([[0, 0, 0, 1]], dtype=points3D.dtype)], dim=0)
    cam = (H4 @ hom.T).T[:, :3]
    z = cam[:, 2]
    front = z > 0
    uv = torch.zeros((n, 2), dtype=points3D.dtype)
    if front.any():
        xn = cam[front] / z[front, None]
        uv[front] = (K[:2, :2] @ xn[:, :2].T).T + K[:2, 2]
    return uv, z


def bilinear_align_corners(depth: np.ndarray, u: np.ndarray, v: np.ndarray) -> np.ndarray:
    """Explicit form of ``grid_sample(bilinear, zeros, align_corners=True)`` as used at
    depth_refiner.py:266-272: bilinear at pixel coordinates (u, v), integer = pixel centre,
    out-of-image taps contribute zero.  Kept in float32 with the same operation order as ATen's
    CPU kernel (bit-identical to ``F.grid_sample`` in tests); the CUDA kernel K1 follows this
    function."""
    h, w = depth.shape
    f32 = np.float32
    gx = (u.astype(f32) / f32(w - 1)) * f32(2) - f32(1)
    gy = (v.astype(f32) / f32(h - 1)) * f32(2) - f32(1)
    ix = ((gx + f32(1)) / f32(2)) * f32(w - 1)
    iy = ((gy + f32(1)) / f32(2)) * f32(h - 1)
    x0 = np.floor(ix)
    y0 = np.floor(iy)
    x1 = x0 + f32(1)
    y1 = y0 + f32(1)
    w_nw = (x1 - ix) * (y1 - iy)
    w_ne = (ix - x0) * (y1 - iy)
    w_sw = (x1 - ix) * (iy - y0)
    w_se = (ix - x0) * (iy - y0)

    def tap(xx, yy):
        ok = (xx >= 0) & (xx <= w - 1) & (yy >= 0) & (yy <= h - 1)
        xi = np.clip(xx, 0, w - 1).astype(np.int64)
        yi = np.clip(yy, 0, h - 1).astype(np.int64)
        return np.where(ok, depth[yi, xi], f32(0)).astype(f32)

    def fma(a, b, c):  # float32 fused multiply-add (product of two float32 is exact in float64)
        return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)

    # ATen's CPU kernel accumulates the taps as a forward FMA chain
    out = fma(tap(x1, y1), w_se, fma(tap(x0, y1), w_sw, fma(tap(x1, y0), w_ne, tap(x0, y0) * w_nw)))
    return out.astype(f32)


def iqr_inliers(z_colmap: torch.Tensor, z_depth: torch.Tensor, outlier_threshold: float) -> torch.Tensor:
    """A3 - depth_refiner.py:117-139.  Lower median, linear-interpolated quartiles, strict <."""
    ratio = z_colmap / (z_depth + 1e-6)
    med = torch.median(ratio)
    q = torch.quantile(ratio, torch.tensor([0.75, 0.25], dtype=torch.float32))
    thr = outlier_threshold * (q[0] - q[1])
    return torch.abs(ratio - med) < thr


def pwl_lookup(d: torch.Tensor, x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """A5 - depth_refiner.py:141-178 ('PCHIP' in name only): piecewise-linear through the pairs
    sorted by x, constant extrapolation, floor at 1e-3.  Knots of equal x keep their pair order (a stable sort, as
    align_stats_kernel sorts): the reference's torch.sort leaves that order to the sort implementation, and a query
    just above a repeated x takes the y of whichever repeat sorts last."""
    if d.numel() < 4:  # depth_refiner.py:143-145 (tests the number of *query pixels*)
        return d * torch.median(y / (d + 1e-6))
    order = torch.argsort(x, stable=True)
    xs = x[order]
    ys = y[order]
    if xs.numel() < 2:
        return d * torch.median(y / (x + 1e-6))
    i = torch.searchsorted(xs, d, right=False).clamp(1, xs.numel() - 1)
    x0, x1, y0, y1 = xs[i - 1], xs[i], ys[i - 1], ys[i]
    dx = x1 - x0
    dx = torch.where(dx == 0, torch.tensor(1e-6, dtype=d.dtype), dx)
    t = ((d - x0) / dx).clamp(0, 1)
    return torch.maximum(y0 + t * (y1 - y0), torch.tensor(1e-3, dtype=d.dtype))


def median3x3_replicate(img: torch.Tensor) -> torch.Tensor:
    """A6 - depth_refiner.py:194-200: 5th smallest of the 3x3 window, replicate border, computed
    over the whole map (zeros at masked pixels participate)."""
    pad = F.pad(img[None, None], (1, 1, 1, 1), mode="replicate")
    win = F.unfold(pad, kernel_size=3).view(9, -1).T
    return torch.median(win, dim=1).values.view(img.shape)


def affine_fit(d: np.ndarray, z: np.ndarray):
    """N1 (parity unpinned): least-squares s, t of z ~ s*d + t from five float64 sums."""
    d = d.astype(np.float64)
    z = z.astype(np.float64)
    n = float(d.size)
    sd, sz, sdd, sdz = d.sum(), z.sum(), (d * d).sum(), (d * z).sum()
    det = n * sdd - sd * sd
    if not det > 0:
        return None
    s = (n * sdz - sd * sz) / det
    t = (sz * sdd - sd * sdz) / det
    return s, t


def refine_view(depth, points3D, cam_from_world, K, mask, cfg: AlignConfig = AlignConfig(), randperm=None):
    """A1-A7 - ``DepthRefiner.refine_depth`` (depth_refiner.py:207-328) on CPU float32.

    ``depth`` [H,W] f32, ``points3D`` [C,3] f64 world, ``cam_from_world`` [3,4] f64, ``K`` [3,3] f64,
    ``mask`` [H,W] bool or None.  ``randperm(n)`` supplies the subsample permutation
    (depth_refiner.py:304).  Returns the reference's dict; early-return paths alias the input."""
    dt = torch.from_numpy(np.ascontiguousarray(depth)).to(torch.float32)
    p3 = torch.from_numpy(np.asarray(points3D)).to(torch.float32)
    T = torch.from_numpy(np.asarray(cam_from_world)).to(torch.float32)
    Kt = torch.from_numpy(np.asarray(K)).to(torch.float32)
    mt = torch.from_numpy(np.asarray(mask)).to(torch.bool) if mask is not None else dt > 0
    h, w = dt.shape
    uv, z = project_sparse(p3, T, Kt)
    m = cfg.edge_margin
    inb = (uv[:, 0] >= m) & (uv[:, 0] < w - m) & (uv[:, 1] >= m) & (uv[:, 1] < h - m) & (z > 0)
    if not inb.any():
        return {"refined_depth": depth, "num_correspondences": 0, "scale_factor": 1.0}
    uvv = uv[inb]
    zc = z[inb]
    grid = torch.stack([uvv[:, 0] / (w - 1) * 2 - 1, uvv[:, 1] / (h - 1) * 2 - 1], dim=-1)[None, None]
    samp = F.grid_sample(dt[None, None], grid, mode="bilinear", padding_mode="zeros", align_corners=True).squeeze()
    if samp.numel() == 0:
        return {"refined_depth": depth, "num_correspondences": 0, "scale_factor": 1.0}
    pos = samp > 0
    if not pos.any():
        return {"refined_depth": depth, "num_correspondences": 0, "scale_factor": 1.0}
    zd = samp[pos]
    zc = zc[pos]
    removed = 0
    if cfg.robust and zd.numel() > 10:  # depth_refiner.py:292 (and :119 - skipped below 10)
        keep = iqr_inliers(zc, zd, cfg.outlier_threshold)
        removed = int((~keep).sum())
        zc, zd = zc[keep], zd[keep]
    if zd.numel() < cfg.min_correspondences:
        return {"refined_depth": depth, "num_correspondences": int(zd.numel()), "scale_factor": 1.0}
    if cfg.align_mode == "pwl" and cfg.adaptive_correspondences and zd.numel() > cfg.max_pairs:
        perm = torch.as_tensor(randperm(zd.numel())) if randperm is not None else torch.randperm(zd.numel())
        idx = perm[: cfg.max_pairs]
        zd, zc = zd[idx], zc[idx]

    out = torch.zeros_like(dt)
    if mt.any():
        if cfg.align_mode == "pwl":
            out[mt] = pwl_lookup(dt[mt], zd, zc)
        else:
            fit = affine_fit(zd.numpy(), zc.numpy())
            if fit is None:
                return {"refined_depth": depth, "num_correspondences": int(zd.numel()), "scale_factor": 1.0}
            s, t = np.float32(fit[0]), np.float32(fit[1])
            out[mt] = torch.clamp(dt[mt] * float(s) + float(t), min=1e-3)
    if not cfg.skip_smoothing:
        out = median3x3_replicate(out)
    out[~mt] = 0
    return {
        "refined_depth": out.numpy().astype(np.float32),
        "num_correspondences": int(zd.numel()),
        "outliers_removed": removed,
        "scale_factor": float(torch.median(zc / (zd + 1e-6))),
    }


# --------------------------------------------------------------------------------------
# Stage 2: back-projection (reference: scripts/test.py:79-90, 194, 205-233)
# --------------------------------------------------------------------------------------
def backproject_view(refined, intr, cam_from_world, stride=1):
    """B1-B3.  ``refined`` already has ``~mask`` zeroed (scripts/test.py:194).  Integer pixel
    coordinates (no half-pixel offset), float32 depth promoted to float64, then
    ``cam_from_world.inverse() * X`` = X R + (-R^T t) row-wise.  Returns world points [Nv,3] f64 and
    the (y, x) pixel indices in row-major order."""
    h, w = refined.shape
    py, px = np.mgrid[0:h:stride, 0:w:stride]
    valid = refined[py, px] > 0
    pxv, pyv = px[valid], py[valid]
    d = refined[pyv, pxv]
    fx, fy, cx, cy = intr
    xn = (pxv - cx) / fx
    yn = (pyv - cy) / fy
    cam = np.stack([xn * d, yn * d, d], axis=-1)
    R = cam_from_world[:, :3]
    t = cam_from_world[:, 3]
    Rinv = R.T
    tinv = -R.T @ t
    world = cam @ Rinv.T + tinv
    return world, pyv, pxv


# --------------------------------------------------------------------------------------
# Stage 3: multi-view consistency votes (reference: scripts/test.py:58-76, 273-333)
# --------------------------------------------------------------------------------------
def project_points(points3d, cam_from_world34, Kmat):
    """C1 - scripts/test.py:58-76: float64, the +1e-8 in the normalisation matters."""
    hom = np.hstack([points3d, np.ones((len(points3d), 1))])
    cam = (cam_from_world34 @ hom.T).T[:, :3]
    z = cam[:, 2]
    xn = cam / (z[:, np.newaxis] + 1e-8)
    uv = (Kmat @ xn.T).T[:, :2]
    return uv, z


def kmatrix(intr):
    fx, fy, cx, cy = intr
    return np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], dtype=np.float64)


def votes_against_view(points, normals, refined_t, cam_from_world_t, intr_t, depth_threshold=0.7, grazing=0.087,
                       sample_mode="nearest", two_sided_tau=None, return_detail=False):
    """C1-C4 for ONE target view: bool vote per point.

    nearest (reference): truncate (u, v) to int, D = refined[vi, ui] (f32), vote iff
    ``z < float32(depth_threshold * D)`` (NEP-50: python float x f32 array stays f32).
    bilinear (N3, parity unpinned): 4 taps at floor(u), floor(v) (+1 clamped), all > 0 required,
    weights of fast_pchip_refiner.py:163-183.  ``two_sided_tau`` switches to |z - D| > tau*D."""
    h, w = refined_t.shape
    uv, z = project_points(points, cam_from_world_t, kmatrix(intr_t))
    R = cam_from_world_t[:, :3]
    c = -R.T @ cam_from_world_t[:, 3]
    dirs = points - c
    dirs /= np.linalg.norm(dirs, axis=1)[:, np.newaxis]
    dots = np.sum(normals * -dirs, axis=1)  # camera-frame normal vs world dir: reference quirk (C2)
    not_grazing = dots > grazing
    u, v = uv[:, 0], uv[:, 1]
    inb = (u >= 0) & (u < w) & (v >= 0) & (v < h) & (z > 0) & not_grazing
    vote = np.zeros(len(points), dtype=bool)
    detail = {"u": u, "v": v, "z": z, "dot": dots, "inb": inb}
    if not inb.any():
        return (vote, detail) if return_detail else vote
    zi = z[inb]
    if sample_mode == "nearest":
        ui = u[inb].astype(int)
        vi = v[inb].astype(int)
        D = refined_t[vi, ui]
        ok = D > 0
    else:
        uu, vv = u[inb], v[inb]
        x0 = np.floor(uu).astype(int)
        y0 = np.floor(vv).astype(int)
        x1 = x0 + 1
        y1 = y0 + 1
        x0c, x1c = np.clip(x0, 0, w - 1), np.clip(x1, 0, w - 1)
        y0c, y1c = np.clip(y0, 0, h - 1), np.clip(y1, 0, h - 1)
        ta, tb, tc, td = refined_t[y0c, x0c], refined_t[y0c, x1c], refined_t[y1c, x0c], refined_t[y1c, x1c]
        ok = (ta > 0) & (tb > 0) & (tc > 0) & (td > 0)
        fx_, fy_ = (uu - x0).astype(np.float32), (vv - y0).astype(np.float32)
        one = np.float32(1)
        D = ((one - fx_) * (one - fy_) * ta + fx_ * (one - fy_) * tb + (one - fx_) * fy_ * tc + fx_ * fy_ * td).astype(np.float32)
    if two_sided_tau is None:
        bad = zi[ok] < depth_threshold * D[ok]
    else:
        bad = np.abs(zi[ok] - D[ok]) > np.float32(two_sided_tau) * D[ok]
    idx = np.where(inb)[0][ok][bad]
    vote[idx] = True
    if return_detail:
        Dfull = np.zeros(len(points), dtype=np.float32)
        Dfull[np.where(inb)[0]] = D
        detail["D"] = Dfull
        return vote, detail
    return vote


def consistency_votes(points, normals, src_view, refined_all, poses, intr, nbr, view_ids=None, **kw):
    """Votes of every point against the neighbour views of its source view.

    ``nbr`` [V,K] int32 (-1 = unused).  With ``nbr = all_views_table`` this is exactly the reference
    loop (scripts/test.py:275-328): every cached view tests every point, own view included."""
    V = refined_all.shape[0]
    votes = np.zeros(len(points), dtype=np.int64)
    member = np.zeros((V, V), dtype=bool)
    for s in range(V):
        for t in nbr[s]:
            if t >= 0:
                member[s, t] = True
    for t in range(V):
        if view_ids is not None and t not in view_ids:
            continue
        sel_views = member[:, t]
        if not sel_views.any():
            continue
        if sel_views.all():
            sel = slice(None)
            pts, nrm = points, normals
        else:
            sel = np.where(sel_views[src_view])[0]
            if len(sel) == 0:
                continue
            pts, nrm = points[sel], normals[sel]
        vt = votes_against_view(pts, nrm, refined_all[t], poses[t], intr[t], **kw)
        votes[sel] += vt
    return votes


# --------------------------------------------------------------------------------------
# Stage 4 (N4/N5, parity unpinned): voxel fusion and sparse merge
# --------------------------------------------------------------------------------------
def voxel_origin(xyz32: np.ndarray, voxel: float) -> np.ndarray:
    """o = floor(bbox_min / voxel) * voxel in float32."""
    v = np.float32(voxel)
    return (np.floor(xyz32.min(axis=0).astype(np.float32) / v) * v).astype(np.float32)


def voxel_keys(xyz32: np.ndarray, voxel: float, origin: np.ndarray) -> np.ndarray:
    """k_axis = int32(floor((p - o) / voxel)) in IEEE float32; key = kx | ky<<21 | kz<<42."""
    v = np.float32(voxel)
    k = np.floor((xyz32.astype(np.float32) - origin.astype(np.float32)) / v).astype(np.int64)
    assert (k >= 0).all() and (k < (1 << 21)).all()
    return (k[:, 0] | (k[:, 1] << 21) | (k[:, 2] << 42)).astype(np.uint64)


def voxel_fuse(xyz32: np.ndarray, rgb: np.ndarray, voxel: float, origin: np.ndarray | None = None):
    """N4: per-voxel count, mean position (float64 accumulation) and round-half-up mean colour.
    Returns keys ascending."""
    if len(xyz32) == 0:
        return (np.zeros(0, np.uint64), np.zeros((0, 3), np.float32), np.zeros((0, 3), np.uint8), np.zeros(0, np.int32))
    if origin is None:
        origin = voxel_origin(xyz32, voxel)
    keys = voxel_keys(xyz32, voxel, origin)
    uk, inv, cnt = np.unique(keys, return_inverse=True, return_counts=True)
    sums = np.zeros((len(uk), 3), dtype=np.float64)
    np.add.at(sums, inv, xyz32.astype(np.float64))
    csum = np.zeros((len(uk), 3), dtype=np.int64)
    np.add.at(csum, inv, rgb.astype(np.int64))
    mean = (sums / cnt[:, None]).astype(np.float32)
    col = ((2 * csum + cnt[:, None]) // (2 * cnt[:, None])).astype(np.uint8)
    return uk, mean, col, cnt.astype(np.int32)


def merge_sparse(sparse_xyz, sparse_rgb, dense_xyz, dense_rgb, dense_keys=None, voxel=None, origin=None, dedup=False):
    """N5 / M1 (scripts/test.py:353-359): sparse points are retained and dense points appended.
    ``dedup`` (new) drops dense voxels whose key is occupied by a sparse point."""
    if dedup:
        s32 = sparse_xyz.astype(np.float32)
        k = np.floor((s32 - origin) / np.float32(voxel)).astype(np.int64)
        inside = ((k >= 0) & (k < (1 << 21))).all(axis=1)
        sk = (k[:, 0] | (k[:, 1] << 21) | (k[:, 2] << 42)).astype(np.uint64)[inside]
        keep = ~np.isin(dense_keys, sk)
        dense_xyz, dense_rgb = dense_xyz[keep], dense_rgb[keep]
    return np.concatenate([sparse_xyz, dense_xyz.astype(np.float64)], 0), np.concatenate([sparse_rgb, dense_rgb], 0)


# --------------------------------------------------------------------------------------
# Whole path
# --------------------------------------------------------------------------------------
def densify(mono_depth, normal, mask, rgb, sparse_xyz, sparse_offsets, poses, intr, nbr, vote_threshold,
            align: AlignConfig = AlignConfig(), depth_threshold=0.7, stride=1, voxel=None, randperm=None,
            sample_mode="nearest", two_sided_tau=None):
    """Stages 1-3 (+4 when ``voxel`` is given) on host arrays, following scripts/test.py:130-333.

    Views without sparse points are skipped entirely (scripts/test.py:136-137): they are neither
    back-projected nor used as filter targets."""
    V, H, W = mono_depth.shape
    refined_all = np.zeros((V, H, W), dtype=np.float32)
    active = []
    stats = []
    pts, cols, nrms, srcs, pix = [], [], [], [], []
    for v in range(V):
        lo, hi = int(sparse_offsets[v]), int(sparse_offsets[v + 1])
        if hi == lo:
            stats.append(None)
            continue
        active.append(v)
        Kmat = kmatrix(intr[v])
        res = refine_view(mono_depth[v].copy(), sparse_xyz[lo:hi], poses[v], Kmat, mask[v], align, randperm)
        ref = np.array(res["refined_depth"], dtype=np.float32, copy=True)
        ref[~mask[v]] = 0  # scripts/test.py:194
        refined_all[v] = ref
        stats.append({k: res[k] for k in res if k != "refined_depth"})
        world, pyv, pxv = backproject_view(ref, intr[v], poses[v], stride)
        pts.append(world)
        cols.append(rgb[v][pyv, pxv])
        nrms.append(normal[v][pyv, pxv])
        srcs.append(np.full(len(world), v, dtype=np.int32))
        pix.append((pyv * W + pxv).astype(np.int64))
    out = {"refined": refined_all, "stats": stats, "active_views": np.array(active, dtype=np.int64)}
    if not pts:
        return out
    points = np.concatenate(pts, 0)
    colors = np.concatenate(cols, 0)
    normals = np.concatenate(nrms, 0)
    src = np.concatenate(srcs, 0)
    votes = consistency_votes(points, normals, src, refined_all, poses, intr, nbr, view_ids=set(active),
                              depth_threshold=depth_threshold, sample_mode=sample_mode, two_sided_tau=two_sided_tau)
    keep = votes < vote_threshold
    out.update(points=points, colors=colors, normals=normals, src_view=src, pixel=np.concatenate(pix, 0),
               votes=votes, keep=keep, counts_per_view=np.array([len(p) for p in pts], dtype=np.int64))
    if voxel is not None:
        xyz32 = points[keep].astype(np.float32)
        origin = voxel_origin(xyz32, voxel) if len(xyz32) else np.zeros(3, np.float32)
        k, m, c, n = voxel_fuse(xyz32, colors[keep], voxel, origin)
        out.update(voxel_origin=origin, voxel_keys=k, voxel_xyz=m, voxel_rgb=c, voxel_count=n)
    return out
