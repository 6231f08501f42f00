"""Hashed voxel fusion (csrc/fuse_hash.cu) at cfg 2 parameters (185 x 1297x840 views, K = 8 nearest, 1 cm voxels,
stride 1), one B200:

  dense     the cfg 2 scene through DensifyEngine.run with the default session (dense occupancy bitmap)
  hashed    the same scene with max_grid_cells = 1 << 16, so the device takes the hashed path; its voxel outputs and
            counts are first asserted bit-identical to `dense`
  dome      a cfg-2-sized scene with distant background (dome_radius 200 m): its box is far beyond 2^35 cells, so only
            the hashed path can fuse it (step time, voxels, grid cells)
  host_grid the host-grid entry points on a grid of more than 2^35 cells, which also fuse through the hashed kernels:
            ops.voxel_fuse over the first 10^4 and 10^6 kept points of the cfg 2 step and over all of them, and
            ops.voxel_fuse_partial on two halves of all kept points followed by ops.voxel_merge_partials

dense and hashed are timed alternately in the same run (`--rounds` pairs).  Step times: CUDA events around `steps`
back-to-back steps after `warmup`; per-stage times: a separate pass with events between align, K4 + fused mark, the
dense finish and the hashed finish (each returns at once when the grid belongs to the other path).  Inputs are
device-resident and far larger than the 126 MB L2.  The card's name, power limit and SM clock are recorded.

  python scripts/gpu/hashed_fuse_bench.py [--steps 10] [--warmup 3] [--rounds 2] [--out profiles/r04_hashed_fuse.json]
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
from depthdensifier_b200.engine import DensifyConfig, DensifyEngine, clamp_vote_threshold  # noqa: E402
from depthdensifier_b200.neighbours import default_vote_threshold, nearest_views_table  # noqa: E402
from depthdensifier_b200.synthetic import SceneConfig, make_scene  # noqa: E402
from ragged_bench import card  # noqa: E402

V, W, H, K, C, VOXEL = 185, 1297, 840, 8, 4096, 0.01
DOME_RADIUS = 200.0


def staged_step(eng: DensifyEngine, sc, nbr, thr) -> dict:
    """The stages of DensifyEngine.run with events between them (a measurement pass, not the timed steps)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    ev[0].record()
    box = ops.new_bbox(sc.cam_from_world.device)
    pair, src = ops.build_pair_tables(sc.cam_from_world, sc.intrinsics, nbr, 0, V, H, W)
    refined, _ = ops.align_views(sc.mono_depth, sc.mask, sc.cam_from_world, ops.intrinsics_matrix(sc.intrinsics), sc.sparse_xyz,
                                 sc.sparse_offsets, C, eng.cfg.align, src_table=src, bbox=box)
    ev[1].record()
    sess = eng.session()
    sess.begin([box], VOXEL)
    xyz, votes = ops.backproject_filter(refined, sc.normal, nbr, pair, src, 0, thr, eng.cfg.filter, bbox=ops.new_bbox(box.device),
                                        mark=sess)
    ev[2].record()
    pts = (xyz.view(-1, 3), sc.rgb.view(-1, 3), votes.view(-1))
    out = ops.fuse_finish(sess, *pts, thr, row_len=W)[:4]
    ev[3].record()
    ops.fuse_finish_hashed(sess, eng.hash_fuse(pts[0].shape[0]), *pts, thr, row_len=W, out=out)
    ev[4].record()
    torch.cuda.synchronize()
    names = ("align", "k4_mark", "dense_finish", "hashed_finish")
    return {n: ev[i].elapsed_time(ev[i + 1]) for i, n in enumerate(names)}


def timed(step, steps: int, warmup: int) -> float:
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="profiles/r04_hashed_fuse.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hashed_fuse_bench needs a CUDA device")
    dev = torch.device("cuda")
    thr = clamp_vote_threshold(default_vote_threshold(K))
    engines = {"dense": DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr), dev),
               "hashed": DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr, max_grid_cells=1 << 16), dev)}
    out = {"card": card(), "workload": f"cfg2 parameters: {V} views at {W}x{H}, K={K}, {VOXEL} m voxels, stride 1",
           "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds}

    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0), device=dev)
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    res = {k: e.run(*inputs) for k, e in engines.items()}
    status = {k: r.session.grid_state() for k, r in res.items()}
    assert status["dense"].status == _lib.GRID_OK and status["hashed"].status == _lib.GRID_HASHED
    for f in ("voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts"):
        assert torch.equal(getattr(res["dense"], f), getattr(res["hashed"], f)), f
    kept_xyz, kept_rgb = res["dense"].kept_points()
    out["check"] = {"dense_vs_hashed": "bit-identical", "kept_points": int(res["dense"].counts[0]), "voxels": int(res["dense"].counts[1]),
                    "grid_cells": int(status["dense"].cells), "hash_buffer_bytes": engines["hashed"]._hash.nbytes(),
                    "hash_cap_points": engines["hashed"]._hash.cap_voxels}
    del res

    times = {k: [] for k in engines}
    stages = {k: [] for k in engines}
    for _ in range(args.rounds):  # alternate the two paths within one run
        for k, e in engines.items():
            times[k].append(timed(lambda: e.run(*inputs, sync=False), args.steps, args.warmup))
            stages[k].append(staged_step(e, sc, nbr, thr))
            stages[k].append(staged_step(e, sc, nbr, thr))
    for k in engines:
        out[k] = {"ms_per_step": times[k], "stages_ms": {s: float(np.median([p[s] for p in stages[k]])) for s in stages[k][0]}}
    # kernels of the hashed finish, from a profiled pass of its own (after the timed ones)
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            engines["hashed"].run(*inputs, sync=False)
        torch.cuda.synchronize()
    dev_ms = lambda e: getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1000.0 / 2
    out["hashed"]["kernels_ms_per_step"] = {e.key.split("(")[0]: dev_ms(e) for e in prof.key_averages() if "hash_" in e.key}

    # host-grid entry points: the same kept points on a host grid of more than 2^35 cells
    lo = kept_xyz.min(0).values.cpu().numpy()
    grid = ops.make_grid(lo, lo + 400.0, VOXEL)
    cells = int(np.prod([grid.dims[i] for i in range(3)], dtype=np.float64))
    assert cells > 2**35
    n_all = int(kept_xyz.shape[0])
    out["host_grid"] = {"grid_cells": cells}
    for n in (10**4, 10**6, n_all):
        fuse = lambda: ops.voxel_fuse(kept_xyz[:n], kept_rgb[:n], None, 1, grid, trim=False)
        out["host_grid"][f"voxel_fuse_{n}"] = {"ms_per_call": timed(fuse, args.steps, args.warmup), "voxels": int(fuse()[4][1])}

    def partials_merge():
        parts = [ops.voxel_fuse_partial(kept_xyz[a:b], kept_rgb[a:b], None, 1, grid) for a, b in ((0, n_all // 2), (n_all // 2, n_all))]
        return ops.voxel_merge_partials(torch.cat([r[: int(c[1])] for r, c in parts]), grid)

    out["host_grid"][f"partials_merge_{n_all}"] = {"ms_per_call": timed(partials_merge, args.steps, args.warmup),
                                                   "voxels": int(partials_merge()[4][1])}
    del kept_xyz, kept_rgb, sc, inputs
    engines["dense"] = None
    torch.cuda.empty_cache()

    dome = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0, dome_radius=DOME_RADIUS), device=dev)
    dnbr = torch.from_numpy(nearest_views_table(dome.cam_from_world.cpu().numpy(), K).astype(np.int32)).to(dev)
    dinputs = (dome.mono_depth, dome.normal, dome.mask, dome.rgb, dome.cam_from_world, dome.intrinsics, dome.sparse_xyz,
               dome.sparse_offsets, dnbr)
    deng = DensifyEngine(DensifyConfig(voxel=VOXEL, vote_threshold=thr), dev)
    r = deng.run(*dinputs)
    st = r.session.grid_state()
    assert st.status == _lib.GRID_HASHED
    out["dome"] = {"dome_radius_m": DOME_RADIUS, "grid_cells": int(st.cells), "dims": list(st.dims), "voxels": r.check(),
                   "kept_points": int(r.counts[0]), "ms_per_step": timed(lambda: deng.run(*dinputs, sync=False), args.steps, args.warmup)}
    out["card_after"] = card()
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
