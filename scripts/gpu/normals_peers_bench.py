"""Cost of the multi-GPU fused normals (the *_normals forms of the dense and hashed peer merges) on ONE B200 with VIRTUAL
ranks: a scene is run once on one GPU with DensifyConfig.fuse_normals (DensifyEngine.run), then its kept points and
per-point normals are dealt to R = 2, 4, 8 ranks in contiguous view blocks (shard_bounds) and fused by R sessions in this
process, whose local addresses stand in for the peers' NVLink mappings.  The plain form (48-byte records) and the
normals form (80-byte records), each on its own sessions, alternate in every round; both concatenations are asserted
bit-identical to the one-GPU result, the voxel normals included.

Workloads: cfg 2 (185 views at 1297x840, K = 8, 1 cm voxels, stride 1: the dense session merge) and the cfg 2-sized
dome scene (dome_radius 200 m: a grid beyond 2^35 cells, the hashed merge).  Per R, form and rank: the point-normals pass
on the rank's views, the partial (dense: rank + accumulate into records; hashed: insert, compact, sort to records), the
owner's merge (CUDA events around each call) and, from a separate profiled pass, the pull kernel's time and the record
bytes it moved.  The pull reads LOCAL HBM here, not NVLink.  Inputs are far larger than the 126 MB L2.  The card's name,
power limit and SM clock are recorded.

  python scripts/gpu/normals_peers_bench.py [--rounds 3] [--out profiles/r12_fused_normals_peers.json]
"""

from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from depthdensifier_b200 import _lib, ops  # noqa: E402
from depthdensifier_b200.distributed import shard_bounds  # noqa: E402
from depthdensifier_b200.engine import DensifyConfig, DensifyEngine, clamp_vote_threshold  # noqa: E402
from depthdensifier_b200.neighbours import default_vote_threshold, nearest_views_table  # noqa: E402
from depthdensifier_b200.synthetic import SceneConfig, make_scene  # noqa: E402
from ragged_bench import card  # noqa: E402

V, W, H, K, C, VOXEL, DOME_RADIUS = 185, 1297, 840, 8, 4096, 0.01, 200.0
PULL = ("merge_pull_mark", "hash_pull")
GATHER = ("merge_gather_prefix", "hash_merge_gather")


class Ranks:
    """R virtual ranks of one form (``normals``: 80-byte records) with their own sessions, hash buffers (hashed form),
    records and outputs: the session and the hash buffers keep the scratch of one record width each."""

    def __init__(self, R, n_max, dev, hashed, normals):
        self.R, self.hashed, self.normals = R, hashed, normals
        self.cap = max(ops.hashed_merge_capacity(n_max, R), n_max + 24576 * R + 1024)
        self.sessions = [ops.FuseSession(dev, max_cells=1 << 20 if hashed else 1 << 33, tile_prefix=True) for _ in range(R)]
        self.hfs = [ops.HashFuse(dev, max(n_max, self.cap)) for _ in range(R)] if hashed else None
        self.samples = [ops.new_hash_samples(dev) for _ in range(R)]
        self.plans = [torch.zeros(64, dtype=torch.int64, device=dev) for _ in range(R)]
        width = _lib.RECORD_NORMAL_WORDS if normals else _lib.RECORD_WORDS
        self.records = [torch.empty((n_max, width), dtype=torch.int64, device=dev) for _ in range(R)]
        self.outs = [ops.new_voxel_outputs(self.cap, dev, normals=normals) for _ in range(R)]

    def step(self, parts, thr, box, timing=None):
        ev = lambda: torch.cuda.Event(enable_timing=True)
        marks = []
        for r, (x, c, v, n) in enumerate(parts):
            sess = self.sessions[r]
            sess.begin([box], VOXEL)
            kw = {"normal": n} if self.normals else {}
            if not self.hashed:
                sess.mark_points(x, v, thr)
            a, b = ev(), ev()
            a.record()
            if self.hashed:
                ops.fuse_finish_hashed_partial(sess, self.hfs[r], x, c, v, thr, self.records[r], self.samples[r], row_len=W, **kw)
            else:
                ops.fuse_finish_partial(sess, x, c, v, thr, self.records[r], row_len=W, **kw)
            b.record()
            marks.append((a, b))
        pr = [t.data_ptr() for t in self.records]
        for r in range(self.R):
            a, b = ev(), ev()
            a.record()
            if self.hashed:
                ops.fuse_merge_hashed_peers(self.sessions[r], self.hfs[r], r, self.R, pr, [t.data_ptr() for t in self.samples], self.plans[r],
                                            self.cap, out=self.outs[r], normals=self.normals)
            else:
                ops.fuse_merge_peers(self.sessions[r], r, self.R, pr, [s.tile_prefix.data_ptr() for s in self.sessions], self.plans[r],
                                     self.cap, out=self.outs[r], normals=self.normals)
            b.record()
            marks.append((a, b))
        torch.cuda.synchronize()
        if timing is not None:
            ms = [a.elapsed_time(b) for a, b in marks]
            timing["partial"].append(ms[: self.R])
            timing["merge"].append(ms[self.R:])

    def result(self):
        mv = [int(s.counts[1]) for s in self.sessions]
        return [torch.cat([o[i][:m] for o, m in zip(self.outs, mv)]) for i in range(5 if self.normals else 4)]


def pull_ms(prof, R) -> list[float]:
    """Per rank: the pull kernel's time (ms) in the profiled pass (kernels in launch order, one gather per merge)."""
    rows = []
    for e in prof.events():
        if getattr(e, "device_type", None) != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name.split("(")[0].replace("void ", "").replace("ddn::", "")
        ms = getattr(e, "device_time", getattr(e, "cuda_time", 0.0)) / 1000.0
        if name.startswith(GATHER):
            rows.append(0.0)
        elif rows and name.startswith(PULL):
            rows[-1] += ms
    return rows[-R:]


def normals_ms(sc, res, bounds, rounds) -> list[float]:
    """Per rank: ops.point_normals over the rank's own views (median of ``rounds``)."""
    out = []
    for lo, hi in bounds:
        args = (sc.normal[lo:hi], sc.cam_from_world[lo:hi].contiguous(), sc.intrinsics[lo:hi].contiguous(), res.votes[lo:hi], 1)
        buf = ops.point_normals(*args)
        ts = []
        for _ in range(rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.point_normals(*args, out=buf)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        out.append(float(np.median(ts)))
    return out


def workload(dome, ranks, rounds, dev) -> dict:
    from torch.profiler import ProfilerActivity, profile

    thr = clamp_vote_threshold(default_vote_threshold(K))
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0, dome_radius=DOME_RADIUS if dome else None), device=dev)
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    eng = DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr, fuse_normals=True), dev)
    res = eng.run(*inputs)
    st = res.session.grid_state()
    assert st.status == (_lib.GRID_HASHED if dome else _lib.GRID_OK)
    one = (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.voxel_normal)
    flat = (res.xyz.view(-1, 3), sc.rgb.view(-1, 3), res.votes.view(-1), res.normals.view(-1, 3))
    box = res.bbox_valid
    rep = {"grid": "hashed" if dome else "dense", "grid_cells": int(st.cells), "kept_points": int(res.counts[0]), "voxels": int(res.counts[1])}
    del eng
    torch.cuda.empty_cache()
    per_view = H * W
    for R in ranks:
        bounds = shard_bounds(V, R)
        parts = [tuple(t[lo * per_view:hi * per_view] for t in flat) for lo, hi in bounds]
        n_max = max(p[0].shape[0] for p in parts)
        vr = {f: Ranks(R, n_max, dev, dome, f == "on") for f in ("off", "on")}
        for form in ("off", "on"):  # warm-up and check
            vr[form].step(parts, thr, box)
            got = vr[form].result()
            for x, y in zip(got, one):
                assert torch.equal(x, y), form
        timing = {f: {"partial": [], "merge": []} for f in ("off", "on")}
        for _ in range(rounds):
            for form in ("off", "on"):  # alternated, so drift hits both forms alike
                vr[form].step(parts, thr, box, timing[form])
        row = {"check": "bit-identical to one GPU (normals included)", "points_per_rank": [int(p[0].shape[0]) for p in parts],
               "point_normals_ms": normals_ms(sc, res, bounds, rounds)}
        med = lambda rows: [float(np.median([x[r] for x in rows])) for r in range(R)]
        for form in ("off", "on"):
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                vr[form].step(parts, thr, box)
            received = [int(p[2]) for p in vr[form].plans]
            rec_bytes = 8 * (_lib.RECORD_NORMAL_WORDS if form == "on" else _lib.RECORD_WORDS)
            pull = pull_ms(prof, R)
            row[form] = {"record_bytes": rec_bytes, "partial_ms": med(timing[form]["partial"]), "merge_ms": med(timing[form]["merge"]),
                         "pull_ms": pull, "received_records": received, "pull_bytes": [n * rec_bytes for n in received],
                         "pull_GBps": [n * rec_bytes / (ms * 1e6) if ms > 0 else None for n, ms in zip(received, pull)]}
        row["pull_bytes_ratio"] = sum(row["on"]["pull_bytes"]) / max(sum(row["off"]["pull_bytes"]), 1)
        rep[f"R{R}"] = row
        del vr, parts
        torch.cuda.empty_cache()
    return rep


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ranks", default="2,4,8")
    ap.add_argument("--out", default="profiles/r12_fused_normals_peers.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normals_peers_bench needs a CUDA device")
    dev = torch.device("cuda")
    ranks = [int(x) for x in args.ranks.split(",")]
    out = {"card": card(), "workload": f"{V} views at {W}x{H}, K={K}, {VOXEL} m voxels, stride 1; R virtual ranks on one GPU; "
           f"cfg2: the dense session merge, dome (dome_radius {DOME_RADIUS} m): the hashed merge", "rounds": args.rounds,
           "note": "virtual ranks: the pull reads local HBM, not NVLink; off = 48-byte records, on = 80-byte records with normals"}
    out["cfg2"] = workload(False, ranks, args.rounds, dev)
    out["dome"] = workload(True, ranks, args.rounds, dev)
    out["card_after"] = card()
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
