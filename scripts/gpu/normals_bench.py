"""The fused normals (DensifyConfig.fuse_normals) at cfg 2 (185 synthetic views at 1297x840, K = 8, 1 cm voxels), one B200,
nearest sampling:

  step     the whole DensifyEngine step with fuse_normals off and on, alternating sample by sample
  normals  ddn_point_normals alone on the step's votes (25 B per grid point: votes, the normal map at the pixel, the output)
  fusion   ddn_fuse_finish (rank + accumulate + finalise) against ddn_fuse_finish_normals on the same marked session, with a
           per-kernel split from the library's launch profiler (ddn_profile_enable) in a separate pass

Times are medians of N CUDA-event samples, the modes alternating in one process; the step's working set (>= 3.9 GB) is
far larger than the 126 MB L2.  The card's name and power limit are read in the same call.

  python scripts/gpu/normals_bench.py [--samples 15] [--out profiles/r11_fused_normals.json]
"""

from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts" / "gpu"))

from bench import VOXEL, WORKLOADS  # noqa: E402
from depthdensifier_b200 import _lib, ops  # noqa: E402
from depthdensifier_b200.engine import DensifyConfig, DensifyEngine  # noqa: E402
from depthdensifier_b200.neighbours import nearest_views_table  # noqa: E402
from depthdensifier_b200.synthetic import SceneConfig, make_scene  # noqa: E402
from ragged_bench import card  # noqa: E402
from support_bench import hbm_peak, timed  # noqa: E402


def med(v) -> float:
    return float(np.median(v))


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=15)
    ap.add_argument("--out", default="profiles/r11_fused_normals.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("normals_bench needs a CUDA device")
    card0 = card()
    V, W, H, K, C, desc = WORKLOADS["cfg2"]
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0), device="cuda")
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).cuda()
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    engines = {"off": DensifyEngine(DensifyConfig(voxel=VOXEL), "cuda"), "on": DensifyEngine(DensifyConfig(voxel=VOXEL, fuse_normals=True), "cuda")}
    res = {k: e.run(*inputs) for k, e in engines.items()}
    off, on = res["off"], res["on"]
    for name in ("refined", "votes", "xyz", "voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts"):
        assert torch.equal(getattr(off, name), getattr(on, name)), name
    n_vox = on.check()
    lens = torch.linalg.norm(on.voxel_normal, dim=1)
    unit = float(((lens - 1).abs() <= 1e-6).float().mean())

    # stage timers on the "on" step's session (its marks stay in place: every finish re-ranks the same occupancy)
    sess = engines["on"].session()
    points = (on.xyz.view(-1, 3), on.grid_rgb().view(-1, 3), on.votes.view(-1))
    thr = on.fusion_threshold()
    normal = on.normals.view(-1, 3)
    nout = ops.point_normals(sc.normal, sc.cam_from_world, sc.intrinsics, on.votes, 1)
    assert torch.equal(nout, on.normals)
    cap = points[0].shape[0]
    outs = ops.new_voxel_outputs(cap, torch.device("cuda"), normals=True)
    stages = {
        "point_normals": lambda: ops.point_normals(sc.normal, sc.cam_from_world, sc.intrinsics, on.votes, 1, out=nout),
        "fuse_finish": lambda: ops.fuse_finish(sess, *points, thr, row_len=W, out=outs[:4]),
        "fuse_finish_normals": lambda: ops.fuse_finish(sess, *points, thr, row_len=W, out=outs, normal=normal),
    }
    times = {k: [] for k in stages}
    steps = {k: [] for k in engines}
    for _ in range(3):  # warm-up of every shape
        for f in stages.values():
            f()
        for e in engines.values():
            e.run(*inputs, sync=False)
    torch.cuda.synchronize()
    for _ in range(args.samples):
        for k, f in stages.items():
            times[k].append(timed(f))
        for k, e in engines.items():
            steps[k].append(timed(lambda: e.run(*inputs, sync=False)))
    assert torch.equal(outs[4][:n_vox], on.voxel_normal)

    # per-kernel split of the two finishes (launch profiler: an event after every launch), separate pass
    split = {}
    for k in ("fuse_finish", "fuse_finish_normals"):
        rows = {}
        for _ in range(args.samples):
            _lib.profile(True)
            stages[k]()
            for name, ms in _lib.profile_report():
                rows.setdefault(name, []).append(ms)
            _lib.profile(False)
        split[k] = {name: med(v) for name, v in rows.items()}

    n_grid = on.votes.numel()
    n_valid = on.num_points()
    pn_ms = med(times["point_normals"])
    peak, peak_src = hbm_peak()
    out = {
        "card": card0, "workload": desc, "samples": args.samples,
        "grid_points": n_grid, "valid_points": n_valid, "kept_points": int(on.counts[0]), "voxels": n_vox,
        "voxel_normals_unit_fraction": unit,
        "step_ms": {k: med(v) for k, v in steps.items()},
        "step_spread_ms": {k: [float(np.min(v)), float(np.max(v))] for k, v in steps.items()},
        "stage_ms": {k: med(v) for k, v in times.items()},
        "stage_spread_ms": {k: [float(np.min(v)), float(np.max(v))] for k, v in times.items()},
        "finish_kernel_ms": split,
        "point_normals_bytes": 25 * n_grid,
        "point_normals_gbs": 25 * n_grid / (pn_ms * 1e-3) / 1e9,
        "point_normals_roofline_frac": 25 * n_grid / (pn_ms * 1e-3) / 1e9 / peak,
        "peak_gbs": peak, "peak_source": peak_src,
    }
    out["card_after"] = card()
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
