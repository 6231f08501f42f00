"""Hashed multi-GPU fusion (csrc/fuse_hash_peers.cu) at cfg 2 dome scale on ONE B200 with VIRTUAL ranks: the dome scene
(dome_radius 200 m, 185 views at 1297x840, K = 8 nearest, 1 cm voxels, stride 1; its box is far beyond 2^35 cells) is
fused once on one GPU (DensifyEngine.run, the hashed path), then its kept points are dealt to R = 2, 4, 8 ranks in
contiguous view blocks (shard_bounds) and fused by R sessions and hash buffers in this process, whose local addresses
stand in for the peers' NVLink mappings.  The rank-ordered concatenation is asserted bit-identical to the one-GPU result.

Per R and rank: the partial (insert, compact, sort to records) and the owner's merge, timed with CUDA events around each
call; a separate profiled pass splits the merge into plan (gather, split, cut, plan kernels), pull and merge (insert,
compact, sort + finalise).  The pull reads LOCAL HBM here, not NVLink.  Inputs are far larger than the 126 MB L2.  The
card's name, power limit and SM clock are recorded.

  python scripts/gpu/hashed_peers_bench.py [--rounds 3] [--out profiles/r05_hashed_peers.json]
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
PLAN = ("hash_merge_gather", "hash_merge_split", "hash_merge_cut", "hash_merge_plan")
MERGE = ("hash_merge_insert", "hash_compact", "hash_merge_finalize")


class Ranks:
    def __init__(self, R, n_max, dev):
        self.R = R
        self.cap = ops.hashed_merge_capacity(n_max, R)
        self.sessions = [ops.FuseSession(dev, max_cells=1 << 20) for _ in range(R)]
        self.hfs = [ops.HashFuse(dev, max(n_max, self.cap)) for _ in range(R)]
        self.records = [torch.empty((n_max, 6), dtype=torch.int64, device=dev) for _ in range(R)]
        self.samples = [ops.new_hash_samples(dev) for _ in range(R)]
        self.plans = [torch.zeros(64, dtype=torch.int64, device=dev) for _ in range(R)]
        self.outs = [ops.new_voxel_outputs(self.cap, dev) for _ in range(R)]

    def step(self, parts, thr, box, timing=None):
        ev = lambda: torch.cuda.Event(enable_timing=True)
        marks = []
        for r, (x, c, v) in enumerate(parts):
            self.sessions[r].begin([box], VOXEL)
            a, b = ev(), ev()
            a.record()
            ops.fuse_finish_hashed_partial(self.sessions[r], self.hfs[r], x, c, v, thr, self.records[r], self.samples[r], row_len=W)
            b.record()
            marks.append((a, b))
        pr = [t.data_ptr() for t in self.records]
        ps = [t.data_ptr() for t in self.samples]
        for r in range(self.R):
            a, b = ev(), ev()
            a.record()
            ops.fuse_merge_hashed_peers(self.sessions[r], self.hfs[r], r, self.R, pr, ps, self.plans[r], self.cap, out=self.outs[r])
            b.record()
            marks.append((a, b))
        torch.cuda.synchronize()
        if timing is not None:
            ms = [a.elapsed_time(b) for a, b in marks]
            timing["partial"].append(ms[: self.R])
            timing["merge"].append(ms[self.R:])

    def result(self):
        mv = [int(s.counts[1]) for s in self.sessions]
        return [torch.cat([o[i][:m] for o, m in zip(self.outs, mv)]) for i in range(4)]


def kernel_split(prof, R) -> list[dict]:
    """Per rank: plan / pull / merge kernel time (ms) of the merge, from the profiled pass (kernels in launch order)."""
    rows, cur = [], None
    for e in prof.events():
        if getattr(e, "device_type", None) != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name.split("(")[0].replace("void ", "").replace("ddn::", "")
        ms = getattr(e, "device_time", getattr(e, "cuda_time", 0.0)) / 1000.0
        if name.startswith("hash_merge_gather"):
            cur = {"plan": 0.0, "pull": 0.0, "merge": 0.0}
            rows.append(cur)
        if cur is None:
            continue
        if name.startswith(PLAN):
            cur["plan"] += ms
        elif name.startswith("hash_pull"):
            cur["pull"] += ms
        elif name.startswith(MERGE):
            cur["merge"] += ms
    return rows[-R:]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ranks", default="2,4,8")
    ap.add_argument("--out", default="profiles/r05_hashed_peers.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hashed_peers_bench needs a CUDA device")
    dev = torch.device("cuda")
    thr = clamp_vote_threshold(default_vote_threshold(K))
    out = {"card": card(), "workload": f"cfg2-sized dome scene: {V} views at {W}x{H}, dome_radius {DOME_RADIUS} m, K={K}, "
           f"{VOXEL} m voxels, stride 1; R virtual ranks on one GPU", "rounds": args.rounds,
           "note": "virtual ranks: the pull reads local HBM, not NVLink"}
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0, dome_radius=DOME_RADIUS), device=dev)
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    eng = DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr), dev)
    res = eng.run(*inputs)
    st = res.session.grid_state()
    assert st.status == _lib.GRID_HASHED
    one = (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count)
    flat = (res.xyz.view(-1, 3), sc.rgb.view(-1, 3), res.votes.view(-1))
    box = res.bbox_valid
    per_view = H * W
    # one-GPU hashed finish of the same points, for scale
    sess1, hf1 = eng.session(), eng._hash
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    one_ms, one_out = [], ops.new_voxel_outputs(flat[0].shape[0], dev)
    for _ in range(args.rounds + 1):
        sess1.begin([box], VOXEL)
        a.record()
        ops.fuse_finish_hashed(sess1, hf1, *flat, thr, row_len=W, out=one_out)
        b.record()
        torch.cuda.synchronize()
        one_ms.append(a.elapsed_time(b))
    out["one_gpu"] = {"grid_cells": int(st.cells), "kept_points": int(res.counts[0]), "voxels": int(res.counts[1]),
                      "hashed_finish_ms": one_ms[1:]}
    del eng, sess1, hf1
    torch.cuda.empty_cache()
    from torch.profiler import ProfilerActivity, profile

    for R in [int(x) for x in args.ranks.split(",")]:
        bounds = shard_bounds(V, R)
        parts = [tuple(t[lo * per_view:hi * per_view] for t in flat) for lo, hi in bounds]
        n_max = max(p[0].shape[0] for p in parts)
        vr = Ranks(R, n_max, dev)
        vr.step(parts, thr, box)  # warm-up
        got = vr.result()
        for x, y in zip(got, one):
            assert torch.equal(x, y)
        timing = {"partial": [], "merge": []}
        for _ in range(args.rounds):
            vr.step(parts, thr, box, timing)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            vr.step(parts, thr, box)
        received = [int(p[2]) for p in vr.plans]
        med = lambda rows: [float(np.median([row[r] for row in rows])) for r in range(R)]
        out[f"R{R}"] = {"check": "bit-identical to one GPU", "points_per_rank": [int(p[0].shape[0]) for p in parts],
                        "records_per_rank": [int(t[-1]) for t in vr.samples],
                        "partial_ms": med(timing["partial"]), "merge_ms": med(timing["merge"]), "merge_split_ms": kernel_split(prof, R),
                        "received_records": received, "imbalance": max(received) / (sum(received) / R),
                        "owner_capacity": vr.cap, "voxels_per_rank": [int(s.counts[1]) for s in vr.sessions]}
        del vr, parts
        torch.cuda.empty_cache()
    out["card_after"] = card()
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
