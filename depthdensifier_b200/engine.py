"""Batched device pipeline: align -> back-project + consistency vote -> voxel fusion.

This is the array-level form of the reference's ``main`` hot loops (scripts/test.py:130-333) for a
whole scene at once: structure-of-arrays inputs resident in HBM, one kernel per stage over all
views, no per-view host round trips."""

from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import torch

from . import ops
from .neighbours import default_vote_threshold


@dataclass
class DensifyConfig:
    align: ops.AlignOptions = field(default_factory=lambda: ops.AlignOptions(zero_unmasked_passthrough=True))
    filter: ops.FilterOptions = field(default_factory=ops.FilterOptions)
    vote_threshold: int | None = None  # None -> ceil(K/2); the reference default 5 assumes K = V
    voxel: float | None = 0.01  # None -> no fusion (reference behaviour: keep every point)
    max_grid_cells: int = 1 << 33  # capacity of the fusion session's occupancy bitmap (16 bytes per 96 cells)
    dedup_sparse: bool = False  # N5: no dense voxel where the sparse cloud already has a point (reference: plain append)
    # ShardedDensifier.run only: stage 1 of a step runs on its own stream and may start while the previous step is still
    # fusing / merging (its NVLink-bound exchange leaves the SMs idle).  The caller's inputs must then be complete when
    # run() is called - they are not ordered against work the caller queued on the current stream just before.
    overlap_align: bool = False
    # Multi-view support (parity unpinned): keep a point only when at least min_support neighbour views see its surface
    # within the relative depth error support_tau, |z - D| <= support_tau * D.  None: off (reference behaviour);
    # 0: count support (DensifyResult.support) without dropping anything.
    min_support: int | None = None
    support_tau: float = 0.01
    # With min_support: a neighbour supports a point only when, besides, the round trip source -> neighbour -> source
    # (MVSNet's forward-backward reprojection) lands within support_reproj_px pixels of the point's pixel.  None: no
    # such test.
    support_reproj_px: float | None = None
    # Oriented normals (one GPU): the step also computes every grid point's world-frame normal from the normal maps
    # (DensifyResult.normals, turned toward its camera) and, with fusion, each voxel's fused normal
    # (DensifyResult.voxel_normal).  Off: the normal maps only feed the grazing gate.
    fuse_normals: bool = False

    def __post_init__(self):
        self._check_reproj()

    def _check_reproj(self):
        rho = self.support_reproj_px
        if rho is None:
            return
        if self.min_support is None:
            raise ValueError("support_reproj_px needs min_support")
        if not (math.isfinite(float(rho)) and float(rho) > 0):
            raise ValueError(f"support_reproj_px must be positive and finite, got {rho}")

    def support(self) -> tuple[int, float] | tuple[int, float, float] | None:
        """The ``support`` argument of ops.backproject_filter: (min_support, support_tau), with support_reproj_px
        appended when set, or None when off."""
        self._check_reproj()
        if self.min_support is None:
            return None
        base = (int(self.min_support), float(self.support_tau))
        return base if self.support_reproj_px is None else base + (float(self.support_reproj_px),)

    def vote_threshold_for(self, k: int) -> int:
        """The threshold a step with ``k`` neighbours per view votes with (``vote_threshold`` or ceil(k/2), clamped)."""
        return clamp_vote_threshold(self.vote_threshold if self.vote_threshold is not None else default_vote_threshold(k))


def clamp_vote_threshold(thr: int) -> int:
    """Votes are stored as u8, saturated at 254, with 255 = "pixel has no point": a threshold of 255 or more keeps
    every point that exists (and never a pixel without one), 0 or less keeps none."""
    return max(0, min(int(thr), 255))


def max_sparse_count(sparse_offsets) -> int:
    """The most sparse points any view has (at least 1), from the offsets [V+1] (synchronises on a device tensor)."""
    off = sparse_offsets.cpu().numpy()
    return max(int(np.max(np.diff(off))) if len(off) > 1 else 1, 1)


@dataclass
class DensifyResult:
    refined: torch.Tensor  # [V,H,W] f32
    stats: torch.Tensor  # [V,8] i32 raw ddn_view_stats
    xyz: torch.Tensor  # [n_src,Hs,Ws,3] f32 world
    votes: torch.Tensor  # [n_src,Hs,Ws] u8 (255 = no point)
    vote_threshold: int
    bbox: torch.Tensor | None = None  # [6] i32 ordered encoding
    grid: object | None = None
    voxel_keys: torch.Tensor | None = None
    voxel_xyz: torch.Tensor | None = None
    voxel_rgb: torch.Tensor | None = None
    voxel_count: torch.Tensor | None = None
    counts: torch.Tensor | None = None  # [2] i64: fused points, voxels
    session: object | None = None  # ops.FuseSession that produced the voxels (device-resident grid)
    hash: object | None = None  # ops.HashFuse of the step: fused the voxels when the grid was too large for the session
    bbox_valid: torch.Tensor | None = None  # [6] i32: box of every back-projected pixel (the alignment kernel's bound)
    layout: ops.ViewLayout | None = None  # run_views: refined [P], xyz [G,3], votes [G] are flat over the views of this layout
    rgb: torch.Tensor | None = None  # the step's colours: [V,H,W,3] u8, or flat [P,3] u8 over the views of ``layout``
    stride: int = 1  # back-projection grid stride: xyz / votes hold every stride-th row and column
    support: torch.Tensor | None = None  # like votes: supporting neighbours, min(count, 254), 255 = no point (None: off)
    min_support: int | None = None  # the step's DensifyConfig.min_support
    normals: torch.Tensor | None = None  # fuse_normals: like xyz, [n_src,Hs,Ws,3] f32 (flat [G,3] for run_views), unit or 0
    voxel_normal: torch.Tensor | None = None  # fuse_normals with fusion: [M,3] f32 per voxel, unit or 0

    def fusion_threshold(self) -> int:
        """The threshold the vote bytes are tested with (by keep_mask and the fusion passes)."""
        return ops.fusion_threshold(clamp_vote_threshold(self.vote_threshold), self.min_support is not None)

    def per_view(self, name: str) -> list:
        """Per-view views of a flat output of run_views: ``refined`` -> [H_v, W_v], ``xyz`` -> [Hs_v, Ws_v, 3],
        ``votes``, ``support`` -> [Hs_v, Ws_v] (no copy)."""
        if self.layout is None:
            return list(getattr(self, name))
        return self.layout.split(getattr(self, name), grid=name != "refined")

    def keep_mask(self) -> torch.Tensor:
        return (self.votes != 255) & (self.votes < self.fusion_threshold())

    def grid_rgb(self) -> torch.Tensor:
        """The colours on the back-projection grid, in the order of ``xyz``: [V,Hs,Ws,3], or flat [G,3] for run_views."""
        s = self.stride
        if s == 1:
            return self.rgb
        if self.layout is None:
            return self.rgb[:, ::s, ::s].contiguous()
        return torch.cat([r.reshape(-1, 3) for r in self.layout.strided(self.layout.split(self.rgb))], 0)

    def kept_points(self) -> tuple[torch.Tensor, torch.Tensor]:
        """xyz [M,3] f32 and rgb [M,3] u8 of the points the vote keeps, view by view in grid order."""
        keep = self.keep_mask()
        return self.xyz[keep], self.grid_rgb()[keep]

    def kept_normals(self) -> torch.Tensor:
        """normals [M,3] f32 of the points the vote keeps, in the order of kept_points() (needs fuse_normals)."""
        if self.normals is None:
            raise ValueError("the step computed no normals: set DensifyConfig.fuse_normals")
        return self.normals[self.keep_mask()]

    def host_grid(self):
        """The voxel grid as a host struct (synchronises; raises when the device could not build one)."""
        if self.grid is None and self.session is not None:
            self.grid = self.session.host_grid()
        return self.grid

    def check(self) -> int:
        """Synchronises and validates the fusion outputs; returns the number of voxels."""
        if self.counts is None:
            return 0
        if self.session is not None:
            st = self.session.grid_state()
            if st.status == 1:  # no valid point at all
                return 0
            self.host_grid()  # raises on a grid neither path could fuse
            if self.hash is not None:
                self.hash.check()
        mv = ops.checked_voxel_count(self.counts)
        if self.voxel_keys is not None and mv > self.voxel_keys.shape[0]:
            raise ops.DDNError(f"voxel fusion: {mv} voxels exceed the output capacity {self.voxel_keys.shape[0]}")
        return mv

    def num_points(self) -> int:
        return int((self.votes != 255).sum().item())


class DensifyEngine:
    def __init__(self, config: DensifyConfig | None = None, device: str | torch.device = "cuda"):
        if not torch.cuda.is_available():
            raise ops.DDNError("DensifyEngine needs a CUDA device: depthdensifier_b200 has no CPU fallback")
        self.cfg = config or DensifyConfig()
        self.device = torch.device(device)

    def align(self, depth, mask, cam_from_world, intr, sparse_xyz, sparse_offsets, max_sparse_per_view, out=None,
              src_table=None, bbox=None):
        return ops.align_views(depth, mask, cam_from_world, ops.intrinsics_matrix(intr), sparse_xyz, sparse_offsets,
                               max_sparse_per_view, self.cfg.align, out=out, src_table=src_table, bbox=bbox)

    def session(self) -> ops.FuseSession:
        if getattr(self, "_session", None) is None or self._session.max_cells != self.cfg.max_grid_cells:
            self._session = ops.FuseSession(self.device, self.cfg.max_grid_cells)
        return self._session

    def hash_fuse(self, n_points: int) -> ops.HashFuse:
        """The hashed fusion path's buffers, grown when a step has more points (+ dedup points) than they hold."""
        if getattr(self, "_hash", None) is None or self._hash.cap_voxels < n_points:
            self._hash = None  # free the old buffers first
            self._hash = ops.HashFuse(self.device, n_points)
        return self._hash

    def run(self, depth, normal, mask, rgb, cam_from_world, intr, sparse_xyz, sparse_offsets, nbr,
            max_sparse_per_view: int | None = None, grid=None, sync: bool = True) -> DensifyResult:
        """All inputs are CUDA tensors: depth [V,H,W] f32, normal [V,H,W,3] f32, mask [V,H,W] bool,
        rgb [V,H,W,3] u8, cam_from_world [V,3,4] f64, intr [V,4] f64, sparse_xyz [S,3] f64,
        sparse_offsets [V+1] i64, nbr [V,K] i32.

        No host round trip between the stages: the voxel grid is derived on the device from the bounding box the
        alignment kernel produces, the consistency kernel marks the occupancy of the points it keeps, and the
        fusion passes read the grid from device memory.  ``sync`` (default): wait at the end, validate
        (``DensifyResult.check()``) and trim the voxel arrays to their count; without it the arrays keep their
        capacity and ``counts`` [2] on the device says how many entries are valid."""
        return self._step(None, depth, normal, mask, rgb, cam_from_world, intr, sparse_xyz, sparse_offsets, nbr,
                          max_sparse_per_view, grid, sync)

    def run_views(self, depths, normals, masks, rgbs, cam_from_world, intr, sparse_xyz, sparse_offsets, nbr,
                  max_sparse_per_view: int | None = None, grid=None, sync: bool = True,
                  layout: ops.ViewLayout | None = None) -> DensifyResult:
        """``run`` for views of different sizes.  ``depths``, ``normals``, ``masks``, ``rgbs``: lists of per-view CUDA
        tensors ([H_v,W_v] f32, [H_v,W_v,3] f32, [H_v,W_v] bool, [H_v,W_v,3] u8), or, with ``layout``, the flat
        concatenations ([P], [P,3], [P], [P,3]); the other inputs as in ``run``.  ``normals`` may be pinned host memory.

        The same step as ``run`` - one launch per stage over all views, no host round trip - on the flat layout
        (include/ddn_b200.h, DDN_LAYOUT_COLS).  The result's refined [P], xyz [G,3] and votes [G] are flat in view order
        (``DensifyResult.per_view`` splits them); keep_mask() and the voxel outputs mean what they mean for ``run``."""
        if layout is None:
            layout = ops.ViewLayout.from_shapes([tuple(d.shape) for d in depths], self.cfg.filter.stride)
            on_device = normals[0].is_cuda
            depths, normals = layout.flatten(depths, torch.float32), layout.flatten(normals, torch.float32)
            normals = normals if on_device else normals.pin_memory()
            masks = layout.flatten(masks) if masks is not None else None
            rgbs = layout.flatten(rgbs) if rgbs is not None else None
        return self._step(layout, depths, normals, masks, rgbs, cam_from_world, intr, sparse_xyz, sparse_offsets, nbr,
                          max_sparse_per_view, grid, sync)

    def _step(self, layout, depth, normal, mask, rgb, cam_from_world, intr, sparse_xyz, sparse_offsets, nbr,
              max_sparse_per_view, grid, sync) -> DensifyResult:
        """align -> back-project + vote with mark -> fusion over [V,H,W] maps (``layout`` None, the uniform kernels) or
        over the flat maps of ``layout`` (the ragged kernels)."""
        cfg = self.cfg
        dev = cam_from_world.device
        thr = cfg.vote_threshold_for(nbr.shape[1])
        if max_sparse_per_view is None:
            max_sparse_per_view = max_sparse_count(sparse_offsets)
        pair, src = (ops.build_pair_tables(cam_from_world, intr, nbr, 0, *depth.shape) if layout is None
                     else ops.build_pair_tables_ragged(layout, cam_from_world, intr, nbr))
        fuse = cfg.voxel is not None
        box = ops.new_bbox(dev) if fuse and grid is None else None
        args = (depth, mask, cam_from_world, ops.intrinsics_matrix(intr), sparse_xyz, sparse_offsets, max(max_sparse_per_view, 1),
                cfg.align)
        box_args = dict(src_table=src if box is not None else None, bbox=box)
        refined, stats = (ops.align_views(*args, **box_args) if layout is None
                          else ops.align_views_ragged(layout, *args, **box_args))
        sess = None
        if fuse:
            sess = self.session()
            if grid is None:
                sess.begin([box], cfg.voxel)
            else:
                sess.begin_grid(grid)
        bbox = ops.new_bbox(dev)
        extra = {} if cfg.min_support is None else {"support": cfg.support()}
        out = (ops.backproject_filter(refined, normal, nbr, pair, src, 0, thr, cfg.filter, bbox=bbox, mark=sess, **extra)
               if layout is None else
               ops.backproject_filter_ragged(layout, refined, normal, pair, src, thr, cfg.filter, bbox=bbox, mark=sess, **extra))
        xyz, votes = out[:2]
        res = DensifyResult(refined=refined, stats=stats, xyz=xyz, votes=votes, vote_threshold=thr, bbox=bbox, bbox_valid=box,
                            layout=layout, rgb=rgb, stride=cfg.filter.stride, support=out[2] if extra else None,
                            min_support=cfg.min_support)
        thr = res.fusion_threshold()
        if cfg.fuse_normals:
            res.normals = (ops.point_normals(normal, cam_from_world, intr, votes, cfg.filter.stride) if layout is None
                           else ops.point_normals_ragged(layout, normal, cam_from_world, intr, votes))
        if fuse:
            points = (xyz.view(-1, 3), res.grid_rgb().view(-1, 3), votes.view(-1))
            dedup = sparse_xyz.float().contiguous() if cfg.dedup_sparse and sparse_xyz.shape[0] > 0 else None
            if dedup is not None:
                sess.unmark_points(dedup)
            row_len = xyz.shape[2] if layout is None else 0  # 0: the rows differ from view to view
            # Both finishes are enqueued on the same outputs; the device grid decides which one runs (the hashed path
            # takes a grid too large for the session's bitmap, the dense one every other), so nothing is read back.
            nrm = {} if res.normals is None else {"normal": res.normals.view(-1, 3)}
            out = ops.fuse_finish(sess, *points, thr, row_len=row_len, **nrm)[:-1]
            hf = self.hash_fuse(points[0].shape[0] + (0 if dedup is None else dedup.shape[0]))
            *vox, counts = ops.fuse_finish_hashed(sess, hf, *points, thr, row_len=row_len, dedup_xyz=dedup, out=out, **nrm)
            res.session, res.grid, res.hash = sess, grid, hf
            res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count = vox[:4]
            res.voxel_normal = vox[4] if nrm else None
            res.counts = counts.clone()
            if sync:
                mv = res.check()
                res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count = (v[:mv] for v in vox[:4])
                if nrm:
                    res.voxel_normal = vox[4][:mv]
        return res
