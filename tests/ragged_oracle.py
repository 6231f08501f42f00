"""The oracle's whole path (oracle/restatement.py:densify) for views of DIFFERENT sizes.

restatement.densify takes [V,H,W] arrays; the reference itself has no such limit: its main refines each image at that
image's own size (scripts/test.py:145-173) and votes every point against each cached view at that view's size
(:275-328).  This module is the same loop over per-view lists, built only from restatement's per-view functions
(refine_view, backproject_view, votes_against_view, voxel_fuse), which already take each view's size from its own
array.  No reference run with mixed sizes is recorded, so mixed-size parity rests on this restatement;
tests/test_ragged_layout.py checks that it reproduces restatement.densify on a uniform scene."""

from __future__ import annotations

import numpy as np

from oracle import restatement as R


def consistency_votes_views(points, normals, src_view, refined, poses, intr, nbr, view_ids=None, **kw):
    """restatement.consistency_votes with ``refined`` a list of V maps of their own sizes."""
    V = len(refined)
    votes = np.zeros(len(points), dtype=np.int64)
    member = np.zeros((V, V), dtype=bool)
    for s in range(V):
        for t in nbr[s]:
            if t >= 0:
                member[s, t] = True
    for t in range(V):
        if view_ids is not None and t not in view_ids:
            continue
        sel = np.where(member[src_view, t])[0]
        if len(sel) == 0:
            continue
        votes[sel] += R.votes_against_view(points[sel], normals[sel], refined[t], poses[t], intr[t], **kw)
    return votes


def densify_views(mono_depth, normal, mask, rgb, sparse_xyz, sparse_offsets, poses, intr, nbr, vote_threshold,
                  align: R.AlignConfig = R.AlignConfig(), depth_threshold=0.7, stride=1, voxel=None, randperm=None,
                  sample_mode="nearest", two_sided_tau=None):
    """restatement.densify with per-view lists (mono_depth[v] [H_v,W_v], normal[v] [H_v,W_v,3], mask[v], rgb[v]);
    ``refined`` in the output is a list, ``pixel`` the index into the view's own map."""
    V = len(mono_depth)
    refined_all = [np.zeros(np.shape(m), dtype=np.float32) for m in mono_depth]
    active, stats = [], []
    pts, cols, nrms, srcs, pix = [], [], [], [], []
    for v in range(V):
        lo, hi = int(sparse_offsets[v]), int(sparse_offsets[v + 1])
        if hi == lo:  # scripts/test.py:136-137
            stats.append(None)
            continue
        active.append(v)
        res = R.refine_view(np.array(mono_depth[v], copy=True), sparse_xyz[lo:hi], poses[v], R.kmatrix(intr[v]), mask[v], align,
                            randperm)
        ref = np.array(res["refined_depth"], dtype=np.float32, copy=True)
        ref[~mask[v]] = 0  # scripts/test.py:194
        refined_all[v] = ref
        stats.append({k: res[k] for k in res if k != "refined_depth"})
        world, pyv, pxv = R.backproject_view(ref, intr[v], poses[v], stride)
        pts.append(world)
        cols.append(rgb[v][pyv, pxv])
        nrms.append(normal[v][pyv, pxv])
        srcs.append(np.full(len(world), v, dtype=np.int32))
        pix.append((pyv * ref.shape[1] + pxv).astype(np.int64))
    out = {"refined": refined_all, "stats": stats, "active_views": np.array(active, dtype=np.int64)}
    if not pts:
        return out
    points = np.concatenate(pts, 0)
    colors = np.concatenate(cols, 0)
    normals = np.concatenate(nrms, 0)
    src = np.concatenate(srcs, 0)
    votes = consistency_votes_views(points, normals, src, refined_all, poses, intr, nbr, view_ids=set(active),
                                    depth_threshold=depth_threshold, sample_mode=sample_mode, two_sided_tau=two_sided_tau)
    keep = votes < vote_threshold
    out.update(points=points, colors=colors, normals=normals, src_view=src, pixel=np.concatenate(pix, 0),
               votes=votes, keep=keep, counts_per_view=np.array([len(p) for p in pts], dtype=np.int64))
    if voxel is not None:
        xyz32 = points[keep].astype(np.float32)
        origin = R.voxel_origin(xyz32, voxel) if len(xyz32) else np.zeros(3, np.float32)
        k, m, c, n = R.voxel_fuse(xyz32, colors[keep], voxel, origin)
        out.update(voxel_origin=origin, voxel_keys=k, voxel_xyz=m, voxel_rgb=c, voxel_count=n)
    return out
