"""Views of different sizes at cfg 2 parameters (K = 8 nearest views, 1 cm voxels, stride 1), one B200:

  uniform   the cfg 2 scene (185 x 1297x840) through DensifyEngine.run
  ragged    the same scene through DensifyEngine.run_views (flat layout); its refined / stats / votes / xyz / voxel outputs
            are first asserted bit-identical to `uniform`
  mixed     185 views alternating 1297x840 and 840x1297 (same pixel count as cfg 2) through run_views

Each line: whole-step ms (CUDA events around `steps` back-to-back steps after `warmup`) and per-stage ms (a separate
pass with events between align, K4 + fused mark, fusion).  Inputs are device-resident; the per-step working set
(>= 3.9 GB) is far larger than the 126 MB L2.  The card's name, power limit and SM clock are recorded with the numbers.

  python scripts/gpu/ragged_bench.py [--steps 20] [--warmup 3] [--out profiles/r03_ragged_bench.json]
"""

from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))

from depthdensifier_b200 import ops  # noqa: E402
from depthdensifier_b200.engine import DensifyConfig, DensifyEngine, clamp_vote_threshold  # noqa: E402
from depthdensifier_b200.neighbours import default_vote_threshold, nearest_views_table  # noqa: E402
from depthdensifier_b200.synthetic import SceneConfig, make_mixed_scene, make_scene  # noqa: E402

V, W, H, K, C, VOXEL = 185, 1297, 840, 8, 4096, 0.01


def card() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[torch.cuda.current_device()]
        return dict(zip(q.split(","), [x.strip() for x in row.split(",")]))
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(), "error": str(e)}


def staged_step(eng: DensifyEngine, layout, inputs, nbr, thr):
    """The stages of run / run_views with events between them (a measurement pass, not the timed steps)."""
    depth, normal, mask, rgb, poses, intr, sparse, off = inputs
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ev[0].record()
    kmat = torch.zeros((poses.shape[0], 3, 3), dtype=torch.float64, device=poses.device)
    kmat[:, 0, 0], kmat[:, 1, 1], kmat[:, 0, 2], kmat[:, 1, 2], kmat[:, 2, 2] = intr[:, 0], intr[:, 1], intr[:, 2], intr[:, 3], 1.0
    box = ops.new_bbox(poses.device)
    if layout is None:
        pair, src = ops.build_pair_tables(poses, intr, nbr, 0, V, H, W)
        refined, _ = ops.align_views(depth, mask, poses, kmat, sparse, off, C, eng.cfg.align, src_table=src, bbox=box)
    else:
        pair, src = ops.build_pair_tables_ragged(layout, poses, intr, nbr)
        refined, _ = ops.align_views_ragged(layout, depth, mask, poses, kmat, sparse, off, C, eng.cfg.align, src_table=src, bbox=box)
    ev[1].record()
    sess = eng.session()
    sess.begin([box], VOXEL)
    bbox = ops.new_bbox(poses.device)
    if layout is None:
        xyz, votes = ops.backproject_filter(refined, normal, nbr, pair, src, 0, thr, eng.cfg.filter, bbox=bbox, mark=sess)
    else:
        xyz, votes = ops.backproject_filter_ragged(layout, refined, normal, pair, src, thr, eng.cfg.filter, bbox=bbox, mark=sess)
    ev[2].record()
    ops.fuse_finish(sess, xyz.view(-1, 3), rgb.view(-1, 3), votes.view(-1), thr, row_len=W if layout is None else 0)
    ev[3].record()
    torch.cuda.synchronize()
    return {"align": ev[0].elapsed_time(ev[1]), "k4_mark": ev[1].elapsed_time(ev[2]), "fusion": ev[2].elapsed_time(ev[3])}


def measure(step, staged, steps: int, warmup: int) -> dict:
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    torch.cuda.synchronize()
    per = [staged() for _ in range(max(3, steps // 4))]
    return {"ms_per_step": a.elapsed_time(b) / steps, "stages_ms": {k: float(np.median([p[k] for p in per])) for k in per[0]}}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="profiles/r03_ragged_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_bench needs a CUDA device")
    dev = torch.device("cuda")
    thr = clamp_vote_threshold(default_vote_threshold(K))
    eng = DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr), dev)
    out = {"card": card(), "workload": f"cfg2 parameters: {V} views, K={K}, {VOXEL} m voxels, stride 1", "steps": args.steps,
           "warmup": args.warmup}

    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0), device=dev)
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    common = (sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    layout = ops.ViewLayout.from_shapes([(H, W)] * V, 1)
    flat = (sc.mono_depth.view(-1), sc.normal.view(-1, 3), sc.mask.view(-1), sc.rgb.view(-1, 3))

    # outputs first: the ragged path on the uniform scene must give the uniform path's bits
    a = eng.run(sc.mono_depth, sc.normal, sc.mask, sc.rgb, *common)
    b = eng.run_views(*flat, *common, layout=layout)
    assert torch.equal(a.refined.view(-1), b.refined) and torch.equal(a.stats, b.stats)
    assert torch.equal(a.votes.view(-1), b.votes) and torch.equal(a.xyz.view(-1, 3), b.xyz)
    for f in ("voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    out["check"] = {"uniform_vs_ragged": "bit-identical", "valid_pixels": a.num_points(), "voxels": int(a.counts[1])}
    del a, b

    st_inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets)
    out["uniform"] = measure(lambda: eng.run(sc.mono_depth, sc.normal, sc.mask, sc.rgb, *common, sync=False),
                             lambda: staged_step(eng, None, st_inputs, nbr, thr), args.steps, args.warmup)
    ft_inputs = flat + st_inputs[4:]
    out["ragged_uniform_scene"] = measure(lambda: eng.run_views(*flat, *common, layout=layout, sync=False),
                                          lambda: staged_step(eng, layout, ft_inputs, nbr, thr), args.steps, args.warmup)
    del sc, flat, st_inputs, ft_inputs, common
    torch.cuda.empty_cache()

    sizes = [(H, W) if v % 2 == 0 else (W, H) for v in range(V)]
    ms = make_mixed_scene(SceneConfig(n_sparse=C, seed=0), sizes, device=dev)
    mlay = ops.ViewLayout.from_shapes(sizes, 1)
    mflat = (mlay.flatten(ms.mono_depth), mlay.flatten(ms.normal), mlay.flatten(ms.mask), mlay.flatten(ms.rgb))
    mnbr = torch.from_numpy(nearest_views_table(ms.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    mcommon = (ms.cam_from_world, ms.intrinsics, ms.sparse_xyz, ms.sparse_offsets, mnbr)
    r = eng.run_views(*mflat, *mcommon, layout=mlay)
    out["check"]["mixed"] = {"valid_pixels": r.num_points(), "voxels": r.check(), "kept": int(r.counts[0])}
    del r
    out["mixed"] = measure(lambda: eng.run_views(*mflat, *mcommon, layout=mlay, sync=False),
                           lambda: staged_step(eng, mlay, mflat + mcommon[:4], mnbr, thr), args.steps, args.warmup)
    out["card_after"] = card()
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
