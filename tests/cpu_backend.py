"""TEST INFRASTRUCTURE ONLY - a CPU stand-in for ``depthdensifier_b200.ops`` built on the oracle.

It lets the world_size-2 gloo tests drive ``ShardedDensifier`` (halo exchange, bbox all-reduce,
splitter selection, voxel all-to-all, merge) without a GPU.  The voxel partial sums follow the CUDA
kernels' integer fixed-point arithmetic exactly (csrc/fuse.cu), so GPU tests also use
``partial_sums_numpy`` as the bit-exact checker of ``ddn_voxel_partials`` / ``ddn_voxel_merge``."""

from __future__ import annotations

import numpy as np
import torch

from depthdensifier_b200 import ops as _ops
from depthdensifier_b200.hashperm import hash_perm
from oracle import restatement as R

FIX = np.float32(1 << 20)


def grid_tuple(grid):
    return np.float32(grid.voxel), np.array(list(grid.origin), np.float32), list(grid.bits)


def canonical_keys(xyz32, voxel, origin):
    k = np.floor((xyz32 - origin) / voxel).astype(np.int64)
    return k, (k[:, 0] | (k[:, 1] << 21) | (k[:, 2] << 42))


def partial_sums_numpy(xyz32, rgb, voxel, origin):
    """Per-voxel integer sums exactly as the partial-record kernels (accumulate_points_kernel, hash_insert_kernel)
    compute them: keys ascending, the records' words 1..5 before packing."""
    if len(xyz32) == 0:
        z = np.zeros
        return z(0, np.int64), z((0, 3), np.int64), z((0, 3), np.int64), z(0, np.int32)
    k, keys = canonical_keys(xyz32.astype(np.float32), voxel, origin)
    centre = (origin[None] + (k.astype(np.float32) + np.float32(0.5)) * voxel).astype(np.float32)
    fix_scale = np.float32((np.float32(1.0) / np.float32(voxel)) * FIX)  # voxel_fix_scale (csrc/fuse_common.cuh)
    off = np.rint(((xyz32.astype(np.float32) - centre) * fix_scale).astype(np.float32)).astype(np.int64)
    uk, inv, cnt = np.unique(keys, return_inverse=True, return_counts=True)
    sums = np.zeros((len(uk), 3), np.int64)
    np.add.at(sums, inv, off)
    csum = np.zeros((len(uk), 3), np.int64)
    np.add.at(csum, inv, rgb.astype(np.int64))
    return uk, sums, csum, cnt.astype(np.int32)


def pack_records(keys, sums, csum, cnt):
    """The 6-word partial record of include/ddn_b200.h (int64 view of the u64 words)."""
    rec = np.zeros((len(keys), 6), np.int64)
    rec[:, 0] = keys.astype(np.int64)
    rec[:, 1:4] = sums
    c = csum.astype(np.int64)
    rec[:, 4] = (c[:, 0] << 32) | c[:, 1]
    rec[:, 5] = (c[:, 2] << 32) | cnt.astype(np.int64)
    return rec


def unpack_records(rec):
    lo = np.int64(0xFFFFFFFF)
    csum = np.stack([(rec[:, 4] >> 32) & lo, rec[:, 4] & lo, (rec[:, 5] >> 32) & lo], 1)
    return rec[:, 0], rec[:, 1:4], csum, (rec[:, 5] & lo).astype(np.int32)


def finalize_numpy(keys, sums, csum, cnt, voxel, origin):
    kx, ky, kz = keys & 0x1FFFFF, (keys >> 21) & 0x1FFFFF, (keys >> 42) & 0x1FFFFF
    k = np.stack([kx, ky, kz], 1)
    centre = (origin[None] + (k.astype(np.float32) + np.float32(0.5)) * voxel).astype(np.float32)
    inv = np.float64(voxel) / (cnt.astype(np.float64) * float(1 << 20))
    xyz = (centre.astype(np.float64) + sums.astype(np.float64) * inv[:, None]).astype(np.float32)
    c = cnt.astype(np.int64)[:, None]
    col = ((2 * csum + c) // (2 * c)).astype(np.uint8)
    return xyz, col


def merge_numpy(keys, sums, csum, cnt):
    uk, inv = np.unique(keys, return_inverse=True)
    s = np.zeros((len(uk), 3), np.int64)
    np.add.at(s, inv, sums)
    c = np.zeros((len(uk), 3), np.int64)
    np.add.at(c, inv, csum)
    n = np.zeros(len(uk), np.int64)
    np.add.at(n, inv, cnt.astype(np.int64))
    return uk, s, c, n.astype(np.int32)


def _encode(f):
    i = np.asarray(f, np.float32).view(np.int32).copy()
    return np.where(i >= 0, i, i ^ np.int32(0x7FFFFFFF)).astype(np.int32)


class OracleBackend:
    DDNError = _ops.DDNError
    decode_bbox = staticmethod(_ops.decode_bbox)
    make_grid = staticmethod(_ops.make_grid)

    def align_views(self, depth, mask, poses, kmat, sparse, offsets, max_sparse, opts, out=None):
        V = depth.shape[0]
        refined = out if out is not None else torch.empty_like(depth)
        stats = torch.zeros((V, 8), dtype=torch.int32)
        off = offsets.numpy()
        cfg = R.AlignConfig(opts.min_correspondences, opts.edge_margin, opts.robust, opts.outlier_threshold, opts.skip_smoothing,
                            opts.adaptive_correspondences, opts.align_mode, opts.max_pairs)
        for v in range(V):
            lo, hi = int(off[v]), int(off[v + 1])
            m = mask[v].numpy().astype(bool) if mask is not None else None
            d = depth[v].numpy()
            if hi == lo:
                refined[v] = 0
                stats[v, 0] = 5
                continue
            r = R.refine_view(d.copy(), sparse[lo:hi].numpy(), poses[v].numpy(), kmat[v].numpy(), m, cfg,
                              randperm=lambda n: hash_perm(n, opts.subsample_seed))
            ref = np.array(r["refined_depth"], np.float32, copy=True)
            if "outliers_removed" not in r:
                stats[v, 0] = 3
                if opts.zero_unmasked_passthrough:
                    ref[~(m if m is not None else d > 0)] = 0
            stats[v, 1] = r["num_correspondences"]
            refined[v] = torch.from_numpy(ref)
        return refined, stats

    def build_pair_tables(self, poses, intr, nbr, src_begin, n_src, height=0, width=0):
        return (poses.numpy(), intr.numpy(), nbr.numpy()), None

    def new_bbox(self, dev):
        return torch.from_numpy(_encode([np.inf] * 3 + [-np.inf] * 3))

    def backproject_filter(self, refined_all, normal, nbr, pair, src, src_begin, thr, opts, bbox=None, xyz_out=None,
                           votes_out=None):
        poses, intr, _ = pair
        nbr = nbr.numpy()
        ref = refined_all.numpy()
        n_src, H, W = normal.shape[0], ref.shape[1], ref.shape[2]
        s = opts.stride
        Hs, Ws = (H + s - 1) // s, (W + s - 1) // s
        xyz = torch.zeros((n_src, Hs, Ws, 3), dtype=torch.float32)
        votes = torch.full((n_src, Hs, Ws), 255, dtype=torch.uint8)
        lo = np.full(3, np.inf, np.float32)
        hi = np.full(3, -np.inf, np.float32)
        for i in range(n_src):
            world, pyv, pxv = R.backproject_view(ref[src_begin + i], intr[src_begin + i], poses[src_begin + i], s)
            if len(world) == 0:
                continue
            nrm = normal[i].numpy()[pyv, pxv]
            v = np.zeros(len(world), np.int64)
            for t in nbr[i]:
                if t >= 0:
                    v += R.votes_against_view(world, nrm, ref[t], poses[t], intr[t], depth_threshold=opts.depth_threshold,
                                              grazing=opts.grazing_cos, sample_mode=opts.sample_mode,
                                              two_sided_tau=opts.two_sided_tau if opts.two_sided_tau > 0 else None)
            w32 = world.astype(np.float32)
            xyz[i].numpy()[pyv // s, pxv // s] = w32
            votes[i].numpy()[pyv // s, pxv // s] = np.minimum(v, 254).astype(np.uint8)
            kept = w32[v < thr]
            if len(kept):
                lo, hi = np.minimum(lo, kept.min(0)), np.maximum(hi, kept.max(0))
        if bbox is not None:
            enc = _encode(np.concatenate([lo, hi]))
            b = bbox.numpy()
            b[:3] = np.minimum(b[:3], enc[:3])
            b[3:] = np.maximum(b[3:], enc[3:])
        if xyz_out is not None:
            xyz_out.copy_(xyz)
            xyz = xyz_out
        if votes_out is not None:
            votes_out.copy_(votes)
            votes = votes_out
        return xyz, votes

    def _select(self, xyz, rgb, votes, thr, grid):
        voxel, origin, bits = grid_tuple(grid)
        x = xyz.numpy().reshape(-1, 3)
        c = rgb.numpy().reshape(-1, 3)
        sel = votes.numpy().reshape(-1) < thr if votes is not None else np.ones(len(x), bool)
        k = np.floor((x - origin) / voxel)
        inside = ((k >= 0) & (k < np.array([int(d) for d in grid.dims]))).all(1)
        sel = sel & inside
        return x[sel], c[sel], voxel, origin

    CELLS_PER_TILE = 256 * 96  # kOwnUnits * kUnitBits (csrc/fuse.cu)

    def fuse_tile_info(self, grid):
        dims = [int(d) for d in grid.dims]
        cells = dims[0] * dims[1] * dims[2]
        return -(-(-(-cells // 96)) // 256), self.CELLS_PER_TILE

    def _tile_of_keys(self, keys, grid):
        nx, ny = int(grid.dims[0]), int(grid.dims[1])
        k = keys.astype(np.int64)
        cell = (k & 0x1FFFFF) + nx * (((k >> 21) & 0x1FFFFF) + ny * ((k >> 42) & 0x1FFFFF))
        return cell // self.CELLS_PER_TILE

    def voxel_fuse_partial(self, xyz, rgb, votes, thr, grid, row_len=0, tile_prefix=None, out=None):
        x, c, voxel, origin = self._select(xyz, rgb, votes, thr, grid)
        uk, sums, csum, cnt = partial_sums_numpy(x, c, voxel, origin)
        counts = torch.tensor([len(x), len(uk)], dtype=torch.int64)
        if tile_prefix is not None:
            tiles = self._tile_of_keys(uk, grid)
            tile_prefix.copy_(torch.from_numpy(np.searchsorted(tiles, np.arange(tile_prefix.numel())).astype(np.int32)))
        return torch.from_numpy(pack_records(uk, sums, csum, cnt)), counts

    def voxel_merge_partials(self, records, grid, trim=False, tile_range=(0, 0)):
        voxel, origin, _ = grid_tuple(grid)
        rec = records.numpy()
        if tile_range[1] > 0:
            t = self._tile_of_keys(rec[:, 0], grid)
            rec = rec[(t >= tile_range[0]) & (t < tile_range[1])]
        pk, psum, prgb, pcnt = unpack_records(rec)
        uk, s, c, n = merge_numpy(pk, psum, prgb, pcnt)
        xyz, col = finalize_numpy(uk, s, c, n, voxel, origin)
        counts = torch.tensor([len(pk), len(uk)], dtype=torch.int64)
        return torch.from_numpy(uk.astype(np.int64)), torch.from_numpy(xyz), torch.from_numpy(col), torch.from_numpy(n), counts

    def voxel_fuse(self, xyz, rgb, votes, thr, grid, trim=True, row_len=0):
        rec, counts = self.voxel_fuse_partial(xyz, rgb, votes, thr, grid)
        k, x, c, n, _ = self.voxel_merge_partials(rec, grid)
        return k, x, c, n, counts
