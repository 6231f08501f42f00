"""Seeded synthetic COLMAP-like scenes for parity tests and benchmarks.

The scene follows SURVEY.md §8(d): a ground plane z=0 plus three spheres, V cameras on a
jittered ring looking at (0,0,0.5), PINHOLE intrinsics fx=fy=0.8·W, cx=W/2, cy=H/2.  Depth is the
analytic z-depth of the first ray hit (pixel centre at integer coordinates, matching the
reference's ``unproject_points`` convention, /root/reference/scripts/test.py:79-90), the
monocular depth is a per-view scale-distorted copy with 2 % "floater" 8x8 blocks, normals are
analytic in the camera frame, and C sparse points per view are drawn from the surface.

All geometry is evaluated in float64 with torch so the same code runs on the host (tests) and
on the GPU (benchmarks at full BASELINE.json sizes, where host generation would be too slow).
MoGe inference is out of scope (BASELINE.json north_star): these maps stand in for it.
"""

from __future__ import annotations

import math
from dataclasses import dataclass, field, replace

import numpy as np
import torch

SPHERES = ((0.0, 0.0, 0.8, 0.8), (1.5, 0.5, 0.4, 0.4), (-1.2, -0.8, 0.5, 0.5))


@dataclass
class SceneConfig:
    n_views: int = 20
    width: int = 512
    height: int = 384
    n_sparse: int = 4096
    max_depth: float = 20.0
    floater_fraction: float = 0.02
    floater_scale: float = 0.4
    seed: int = 0
    ring_radius: float = 4.0
    ring_height: float = 2.0
    dome_radius: float | None = None
    """Distant background: rays that hit nothing within ``max_depth`` hit the inside of a sphere of this radius around
    the origin (masked in, with analytic normals and colours).  None: no background (those pixels are masked out)."""


@dataclass
class Scene:
    """Structure-of-arrays scene. Tensors live on one device; poses/intrinsics are float64."""

    cfg: SceneConfig
    cam_from_world: torch.Tensor  # [V,3,4] f64
    intrinsics: torch.Tensor  # [V,4] f64 (fx, fy, cx, cy)
    mono_depth: torch.Tensor  # [V,H,W] f32 (MoGe stand-in)
    true_depth: torch.Tensor  # [V,H,W] f32
    normal: torch.Tensor  # [V,H,W,3] f32, camera frame
    mask: torch.Tensor  # [V,H,W] bool
    rgb: torch.Tensor  # [V,H,W,3] u8
    sparse_xyz: torch.Tensor  # [sum C_v, 3] f64 world
    sparse_offsets: torch.Tensor  # [V+1] i64 CSR
    scale: torch.Tensor = field(default=None)  # [V] f64 per-view distortion s_v

    @property
    def n_views(self) -> int:
        return self.cfg.n_views

    def centers(self) -> torch.Tensor:
        R = self.cam_from_world[:, :, :3]
        t = self.cam_from_world[:, :, 3]
        return -(R.transpose(1, 2) @ t.unsqueeze(-1)).squeeze(-1)


def ring_poses(cfg: SceneConfig) -> np.ndarray:
    """[V,3,4] float64 cam_from_world for a jittered ring (COLMAP axes: x right, y down, z fwd)."""
    rng = np.random.default_rng(cfg.seed)
    V = cfg.n_views
    theta = 2.0 * math.pi * np.arange(V) / V
    rad = cfg.ring_radius + rng.uniform(-0.3, 0.3, V)
    hgt = cfg.ring_height + rng.uniform(-0.3, 0.3, V)
    c = np.stack([rad * np.cos(theta), rad * np.sin(theta), hgt], axis=1)
    target = np.array([0.0, 0.0, 0.5])
    fwd = target[None] - c
    fwd /= np.linalg.norm(fwd, axis=1, keepdims=True)
    up = np.array([0.0, 0.0, 1.0])
    right = np.cross(fwd, up[None])
    right /= np.linalg.norm(right, axis=1, keepdims=True)
    down = np.cross(fwd, right)
    R = np.stack([right, down, fwd], axis=1)  # rows
    t = -(R @ c[:, :, None])[:, :, 0]
    return np.concatenate([R, t[:, :, None]], axis=2)


def _raycast(c: torch.Tensor, dw: torch.Tensor, max_depth: float, dome_radius: float | None = None):
    """First hit of rays c + d*dw (d = z-depth since dw = R^T (x, y, 1)). Returns d, n_world, hit.  With
    ``dome_radius``, rays without a hit within ``max_depth`` hit the inside of that sphere around the origin."""
    inf = torch.full(dw.shape[:-1], float("inf"), dtype=dw.dtype, device=dw.device)
    d_plane = torch.where(dw[..., 2] < 0, -c[2] / dw[..., 2].clamp(max=-1e-12), inf)
    best = d_plane
    n = torch.zeros_like(dw)
    n[..., 2] = 1.0
    a = (dw * dw).sum(-1)
    for sx, sy, sz, r in SPHERES:
        s = torch.tensor([sx, sy, sz], dtype=dw.dtype, device=dw.device)
        oc = c - s
        b = (dw * oc).sum(-1)
        cc = (oc * oc).sum() - r * r
        disc = b * b - a * cc
        ok = disc > 0
        d = (-b - torch.sqrt(disc.clamp(min=0))) / a
        ok = ok & (d > 1e-6) & (d < best)
        p = c + d.unsqueeze(-1) * dw
        ns = (p - s) / r
        best = torch.where(ok, d, best)
        n = torch.where(ok.unsqueeze(-1), ns, n)
    hit = torch.isfinite(best) & (best < max_depth) & (best > 0)
    if dome_radius is not None:  # the camera is inside the dome: the far root of |c + d dw| = R
        b = (dw * c).sum(-1)
        disc = b * b - a * ((c * c).sum() - dome_radius * dome_radius)
        d_dome = (-b + torch.sqrt(disc.clamp(min=0))) / a
        dome = ~hit & (disc > 0) & (d_dome > 0)
        best = torch.where(dome, d_dome, best)
        n = torch.where(dome.unsqueeze(-1), -(c + d_dome.unsqueeze(-1) * dw) / dome_radius, n)
        hit = hit | dome
    return best, n, hit


def make_scene(cfg: SceneConfig, device: str | torch.device = "cpu", views: range | None = None) -> Scene:
    """Generate the scene.  ``views`` restricts the per-view maps and sparse points to a sub-range of
    the ``cfg.n_views`` ring (multi-GPU shards, CPU-baseline samples); poses and intrinsics always
    cover the whole ring.  A view's content depends only on (cfg, view index) when the device is
    the same, because each view draws from its own seeded generators."""
    dev = torch.device(device)
    V, H, W = cfg.n_views, cfg.height, cfg.width
    vlist = list(range(V)) if views is None else list(views)
    nv = len(vlist)
    poses_np = ring_poses(cfg)
    poses = torch.from_numpy(poses_np).to(dev)
    fx = fy = 0.8 * W
    cx, cy = W / 2.0, H / 2.0
    intr = torch.tensor([[fx, fy, cx, cy]] * V, dtype=torch.float64, device=dev)

    scale_np = np.random.default_rng(cfg.seed + 1).uniform(0.5, 2.0, V)
    g_float = torch.Generator(device=dev)
    g_sparse = torch.Generator(device=dev)

    mono = torch.empty((nv, H, W), dtype=torch.float32, device=dev)
    true = torch.empty((nv, H, W), dtype=torch.float32, device=dev)
    normal = torch.empty((nv, H, W, 3), dtype=torch.float32, device=dev)
    mask = torch.empty((nv, H, W), dtype=torch.bool, device=dev)
    rgb = torch.empty((nv, H, W, 3), dtype=torch.uint8, device=dev)
    sparse = []
    offsets = [0]

    ys, xs = torch.meshgrid(
        torch.arange(H, dtype=torch.float64, device=dev),
        torch.arange(W, dtype=torch.float64, device=dev),
        indexing="ij",
    )
    dir_cam = torch.stack([(xs - cx) / fx, (ys - cy) / fy, torch.ones_like(xs)], dim=-1)
    bh, bw = (H + 7) // 8, (W + 7) // 8
    for slot, v in enumerate(vlist):
        g_float.manual_seed(cfg.seed * 1000003 + 2 * v + 1)
        g_sparse.manual_seed(cfg.seed * 1000003 + 2 * v + 2)
        R = poses[v, :, :3]
        t = poses[v, :, 3]
        c = -(R.T @ t)
        dw = dir_cam @ R  # rows: R^T dir
        d, n_w, hit = _raycast(c, dw, cfg.max_depth, cfg.dome_radius)
        d = torch.where(hit, d, torch.zeros_like(d))
        n_c = n_w @ R.T
        p_w = c + d.unsqueeze(-1) * dw
        s_v = float(scale_np[v])
        m = d / s_v * (1.0 + 0.05 * torch.sin(d))
        blocks = torch.rand((bh, bw), generator=g_float, device=dev) < cfg.floater_fraction
        fl = blocks.repeat_interleave(8, 0).repeat_interleave(8, 1)[:H, :W]
        m = torch.where(fl, m * cfg.floater_scale, m)
        mono[slot] = torch.where(hit, m, torch.zeros_like(m)).float()
        true[slot] = d.float()
        normal[slot] = torch.where(hit.unsqueeze(-1), n_c, torch.zeros_like(n_c)).float()
        mask[slot] = hit
        q = torch.floor(p_w / 0.05).to(torch.int64)
        hsh = (q[..., 0] * 73856093) ^ (q[..., 1] * 19349663) ^ (q[..., 2] * 83492791)
        rgb[slot] = torch.stack([hsh & 255, (hsh >> 8) & 255, (hsh >> 16) & 255], dim=-1).to(torch.uint8)

        # sparse "COLMAP" points: continuous image positions, exact surface hits, world float64
        ncand = 2 * cfg.n_sparse
        uv = torch.rand((ncand, 2), generator=g_sparse, device=dev, dtype=torch.float64)
        u = uv[:, 0] * (W - 1)
        w_ = uv[:, 1] * (H - 1)
        dc = torch.stack([(u - cx) / fx, (w_ - cy) / fy, torch.ones_like(u)], dim=-1)
        dws = dc @ R
        ds, _, hs = _raycast(c, dws, cfg.max_depth, cfg.dome_radius)
        pts = (c + ds.unsqueeze(-1) * dws)[hs][: cfg.n_sparse]
        sparse.append(pts)
        offsets.append(offsets[-1] + pts.shape[0])

    return Scene(
        cfg=cfg,
        cam_from_world=poses,
        intrinsics=intr,
        mono_depth=mono,
        true_depth=true,
        normal=normal,
        mask=mask,
        rgb=rgb,
        sparse_xyz=torch.cat(sparse, 0) if sparse else torch.zeros((0, 3), dtype=torch.float64, device=dev),
        sparse_offsets=torch.tensor(offsets, dtype=torch.int64, device=dev),
        scale=torch.from_numpy(scale_np).to(dev),
    )


@dataclass
class MixedScene:
    """A scene whose views have different sizes: per-view lists of maps, the other arrays as in ``Scene``."""

    cfg: SceneConfig
    sizes: list  # [(H_v, W_v)]
    cam_from_world: torch.Tensor  # [V,3,4] f64
    intrinsics: torch.Tensor  # [V,4] f64, each view's own (fx = fy = 0.8 W_v, cx = W_v/2, cy = H_v/2)
    mono_depth: list  # V x [H_v,W_v] f32
    normal: list  # V x [H_v,W_v,3] f32
    mask: list  # V x [H_v,W_v] bool
    rgb: list  # V x [H_v,W_v,3] u8
    sparse_xyz: torch.Tensor  # [sum C_v, 3] f64
    sparse_offsets: torch.Tensor  # [V+1] i64

    @property
    def n_views(self) -> int:
        return len(self.sizes)


def make_mixed_scene(cfg: SceneConfig, sizes, device: str | torch.device = "cpu") -> MixedScene:
    """The ring of ``cfg`` (poses from ring_poses(cfg), V = len(sizes)) with view v rendered at sizes[v] = (H_v, W_v):
    its maps and sparse points are those of make_scene(replace(cfg, width=W_v, height=H_v), views=[v]), so a view's
    content depends only on (cfg, v, its size)."""
    cfg = replace(cfg, n_views=len(sizes))
    per = [make_scene(replace(cfg, width=int(w), height=int(h)), device, views=[v]) for v, (h, w) in enumerate(sizes)]
    counts = [sc.sparse_xyz.shape[0] for sc in per]
    return MixedScene(
        cfg=cfg,
        sizes=[(int(h), int(w)) for h, w in sizes],
        cam_from_world=per[0].cam_from_world,
        intrinsics=torch.stack([sc.intrinsics[v] for v, sc in enumerate(per)]),
        mono_depth=[sc.mono_depth[0] for sc in per],
        normal=[sc.normal[0] for sc in per],
        mask=[sc.mask[0] for sc in per],
        rgb=[sc.rgb[0] for sc in per],
        sparse_xyz=torch.cat([sc.sparse_xyz for sc in per], 0),
        sparse_offsets=torch.tensor(np.concatenate([[0], np.cumsum(counts)]), dtype=torch.int64, device=torch.device(device)),
    )
