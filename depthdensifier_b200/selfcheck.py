"""Multi-GPU equivalence check (SURVEY.md §8e criterion): the R-rank sharded pipeline must reproduce the 1-rank
pipeline - refined depth, votes, voxel keys, counts, colours AND positions bit for bit (voxel sums are integer
fixed point).  Runs inside an initialised process group, one rank per GPU; used by bench.py before its timed
region, by scripts/check_multi_gpu.py and by the two-rank GPU test."""

from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from .distributed import ShardedDensifier, shard_bounds
from .engine import DensifyConfig
from .neighbours import nearest_views_table
from .synthetic import SceneConfig, make_scene


def multi_gpu_check(dev, rank: int, world: int, n_views: int = 24, width: int = 320, height: int = 240, k: int = 4,
                    voxel: float = 0.02, steps: int = 2, verbose: bool = False, dedup: bool = False, dome_radius: float | None = None,
                    max_grid_cells: int | None = None, min_support: int | None = None,
                    support_reproj_px: float | None = None, fuse_normals: bool = False) -> dict:
    """Every rank calls this.  Rank 0 returns {"passed": bool, "path": "peer" | "collective", ...}; the other
    ranks the same dict with their local view of ``path``.  ``dome_radius``: the scene gets a distant background
    (SceneConfig.dome_radius), ``max_grid_cells``: the sessions' bitmap capacity - either can send the step through the
    hashed fusion path (``report["grid"]`` says which path fused).  ``min_support``: DensifyConfig.min_support of both
    pipelines (the support counts are then compared too); ``support_reproj_px``: their DensifyConfig.support_reproj_px.
    ``fuse_normals``: DensifyConfig.fuse_normals of both pipelines (the per-point and the voxel normals are then compared
    too, and the voxel normals of run_host)."""
    V, W, H = n_views, width, height
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=1500, seed=4, dome_radius=dome_radius))  # host, identical on all ranks
    nbr = nearest_views_table(sc.cam_from_world.numpy(), k)
    off = sc.sparse_offsets.numpy()

    def inputs(lo, hi, to):
        return (to(sc.mono_depth[lo:hi]), to(sc.normal[lo:hi]), to(sc.mask[lo:hi]), to(sc.rgb[lo:hi]),
                to(sc.sparse_xyz[off[lo]:off[hi]]), to(sc.sparse_offsets[lo:hi + 1] - off[lo]))

    def collect(res):
        mv = res.check()
        return {"keys": res.voxel_keys[:mv].cpu().numpy(), "xyz": res.voxel_xyz[:mv].cpu().numpy(),
                "rgb": res.voxel_rgb[:mv].cpu().numpy(), "count": res.voxel_count[:mv].cpu().numpy(),
                "votes": res.votes.cpu().numpy(), "refined": res.refined.cpu().numpy(), "n": int(res.counts[0]),
                "support": None if res.support is None else res.support.cpu().numpy(),
                "normals": None if res.normals is None else res.normals.cpu().numpy(),
                "normal": None if res.voxel_normal is None else res.voxel_normal[:mv].cpu().numpy()}

    def config(**kw):
        cfg = DensifyConfig(voxel=voxel, dedup_sparse=dedup, min_support=min_support, support_reproj_px=support_reproj_px,
                            fuse_normals=fuse_normals, **kw)
        if max_grid_cells is not None:
            cfg.max_grid_cells = max_grid_cells
        return cfg

    lo, hi = shard_bounds(V, world)[rank]
    sd = ShardedDensifier(config(overlap_align=dedup), dev, rank, world, V, lo, hi, sc.cam_from_world, sc.intrinsics, nbr, H, W)
    path = "peer" if sd.peer is not None else "collective"
    dev_in = inputs(lo, hi, lambda t: t.to(dev).contiguous())
    mine = None
    results = [sd.run(*dev_in) for _ in range(max(steps, 1) + 1)]  # queued back to back: later steps run on reused (and
    mine = collect(results[-1])                                     # cleaned-up) exchange buffers, stage 1 possibly overlapped
    gathered = [None] * world
    dist.gather_object(mine, gathered if rank == 0 else None, dst=0)
    report = {"passed": True, "path": path, "ranks": world, "views": V, "size": [W, H], "steps": steps, "dedup_sparse": dedup, "different": []}
    if min_support is not None:
        report["min_support"] = min_support
    if support_reproj_px is not None:
        report["support_reproj_px"] = support_reproj_px
    if fuse_normals:
        report["fuse_normals"] = True
    if dome_radius is not None or max_grid_cells is not None:
        status = results[-1].session.grid_state().status if results[-1].session is not None else None
        report.update(dome_radius=dome_radius, max_grid_cells=max_grid_cells, grid={0: "dense", 4: "hashed"}.get(status, status))
    one = None
    if rank == 0:
        sd1 = ShardedDensifier(config(), dev, 0, 1, V, 0, V, sc.cam_from_world, sc.intrinsics, nbr, H, W)
        one = collect(sd1.run(*inputs(0, V, lambda t: t.to(dev).contiguous())))
        extra = (() if min_support is None else ("support",)) + (("normals", "normal") if fuse_normals else ())
        for name in ("refined", "votes", "keys", "count", "rgb", "xyz") + extra:
            cat = np.concatenate([g[name] for g in gathered])
            if not np.array_equal(cat, one[name]):
                report["different"].append(name)
        if sum(g["n"] for g in gathered) != one["n"]:
            report["different"].append("n_points")
        report["voxels_per_rank"] = [len(g["keys"]) for g in gathered]
        report["points"] = one["n"]
    # the end-to-end host entry point (pinned host arrays, normals read in place) must give the same cloud
    host = sd.pin_host_inputs(*inputs(lo, hi, lambda t: t.contiguous()))
    out = None
    for _ in range(2):
        out = sd.run_host(*host, chunk_views=5)
    host_names = ("keys", "xyz", "rgb", "count") + (("normal",) if fuse_normals else ())
    mine_h = {name: out[name].numpy().copy() for name in host_names} if "keys" in out else None
    gathered_h = [None] * world
    dist.gather_object(mine_h, gathered_h if rank == 0 else None, dst=0)
    if rank == 0:
        for name in ("keys", "count", "rgb", "xyz") + (("normal",) if fuse_normals else ()):
            parts = [g[name] for g in gathered_h if g is not None]
            if not parts or not np.array_equal(np.concatenate(parts), one[name]):
                report["different"].append("run_host:" + name)
        report["passed"] = not report["different"]
        if verbose:
            print("MULTI-GPU CHECK", "PASSED" if report["passed"] else f"FAILED {report['different']}", report)
    flag = torch.tensor([1 if report["passed"] else 0], device=dev)
    dist.broadcast(flag, src=0)
    report["passed"] = bool(flag.item())
    return report
