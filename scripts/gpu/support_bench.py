"""The multi-view support filter (DensifyConfig.min_support) at cfg 2 (185 synthetic views at 1297x840, K = 8, 1 cm
voxels), one B200, nearest sampling and bilinear as a second line:

  k4     K4 with the fused occupancy mark: the plain kernel against the support form (m = 2, tau = 0.01), same inputs
  step   the whole DensifyEngine step, support off / m = 2 / m = 0
  kept   kept points (counts[0]) and voxels of each mode

--arm reproj (writes profiles/r10_support_reproj.json): the forward-backward reprojection form instead,

  k4     K4 with the fused mark: the support form (m = 2, tau = 0.01) against support + reprojection (rho = 1 px)
  kept   kept points (counts[0]) and voxels of the step at rho in {0.5, 1, 2} and without the reprojection test

Times are medians of N CUDA-event samples, the modes alternating sample by sample in one process.  The step's working set
(>= 3.9 GB) is far larger than the 126 MB L2.  roofline_frac: algorithmic bytes of back-projection + consistency
(29 + 4K = 61 B per valid pixel, as bench.py counts them) over the K4 time, against the HBM peak bench.py uses.  The
card's name and power limit are read in the same call.

  python scripts/gpu/support_bench.py [--samples 15] [--arm support|reproj] [--out PATH]
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
from depthdensifier_b200 import ops  # noqa: E402
from depthdensifier_b200.engine import DensifyConfig, DensifyEngine  # noqa: E402
from depthdensifier_b200.neighbours import nearest_views_table  # noqa: E402
from depthdensifier_b200.synthetic import SceneConfig, make_scene  # noqa: E402
from ragged_bench import card  # noqa: E402

TAU = 0.01


def hbm_peak() -> tuple[float, str]:
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md), as bench.py"


def timed(fn) -> float:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def line(sc, nbr, sample_mode: str, samples: int) -> dict:
    V, H, W = sc.mono_depth.shape
    K = nbr.shape[1]
    modes = {"default": None, "support_m2": 2, "support_m0": 0}
    engines = {k: DensifyEngine(DensifyConfig(voxel=VOXEL, filter=ops.FilterOptions(sample_mode=sample_mode), min_support=m,
                                              support_tau=TAU), "cuda") for k, m in modes.items()}
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    out = {"sample_mode": sample_mode, "modes": {}}
    ref = engines["default"].run(*inputs)
    thr = ref.vote_threshold
    for k, eng in engines.items():
        r = eng.run(*inputs)
        out["modes"][k] = {"min_support": modes[k], "valid_pixels": r.num_points(), "kept_points": int(r.counts[0]),
                           "voxels": r.check()}
        if k == "support_m0":  # m = 0 at thr <= 254: the plain kernel's bytes
            assert torch.equal(r.votes, ref.votes) and torch.equal(r.xyz, ref.xyz) and torch.equal(r.counts, ref.counts)
    n_valid = out["modes"]["default"]["valid_pixels"]

    # K4 with the fused mark on the step's refined maps and grid
    pair, src = ops.build_pair_tables(sc.cam_from_world, sc.intrinsics, nbr, 0, V, H, W)
    sess = ops.FuseSession(torch.device("cuda"))
    grid = ref.host_grid()
    xyz = torch.empty((V, H, W, 3), dtype=torch.float32, device="cuda")
    votes = torch.empty((V, H, W), dtype=torch.uint8, device="cuda")
    sup = torch.empty_like(votes)
    bbox = ops.new_bbox(torch.device("cuda"))
    fopt = engines["default"].cfg.filter

    def k4(support):
        extra = {} if support is None else {"support": support, "support_out": sup}
        return lambda: ops.backproject_filter(ref.refined, sc.normal, nbr, pair, src, 0, thr, fopt, bbox=bbox, xyz_out=xyz,
                                              votes_out=votes, mark=sess, **extra)

    k4s = {"default": k4(None), "support_m2": k4((2, TAU))}
    times = {k: [] for k in k4s}
    steps = {k: [] for k in engines}
    for _ in range(3):  # warm-up of every shape
        for k, f in k4s.items():
            sess.begin_grid(grid)
            f()
        for eng in engines.values():
            eng.run(*inputs, sync=False)
    torch.cuda.synchronize()
    for _ in range(samples):
        for k, f in k4s.items():
            sess.begin_grid(grid)
            times[k].append(timed(f))
        for k, eng in engines.items():
            steps[k].append(timed(lambda: eng.run(*inputs, sync=False)))
    peak, src_peak = hbm_peak()
    bpp = 29 + 4 * K
    med = {k: float(np.median(v)) for k, v in times.items()}
    out["k4_with_mark_ms"] = med
    out["k4_ratio_support_over_default"] = med["support_m2"] / med["default"]
    out["k4_spread_ms"] = {k: [float(np.min(v)), float(np.max(v))] for k, v in times.items()}
    out["roofline_frac"] = {k: bpp * n_valid / (ms * 1e-3) / 1e9 / peak for k, ms in med.items()}
    out["step_ms"] = {k: float(np.median(v)) for k, v in steps.items()}
    out["step_spread_ms"] = {k: [float(np.min(v)), float(np.max(v))] for k, v in steps.items()}
    out["roofline"] = {"algorithmic_bytes_per_pixel": bpp, "peak_gbs": peak, "peak_source": src_peak, "pixels": n_valid}
    return out


def reproj_line(sc, nbr, sample_mode: str, samples: int) -> dict:
    V, H, W = sc.mono_depth.shape
    K = nbr.shape[1]
    fopt = ops.FilterOptions(sample_mode=sample_mode)
    inputs = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    out = {"sample_mode": sample_mode, "min_support": 2, "kept": {}}
    ref = None
    for rho in (None, 0.5, 1.0, 2.0):
        r = DensifyEngine(DensifyConfig(voxel=VOXEL, filter=fopt, min_support=2, support_tau=TAU, support_reproj_px=rho), "cuda").run(*inputs)
        out["kept"]["support_only" if rho is None else f"rho_{rho:g}"] = {
            "support_reproj_px": rho, "valid_pixels": r.num_points(), "kept_points": int(r.counts[0]), "voxels": r.check()}
        ref = r if rho is None else ref
    n_valid = out["kept"]["support_only"]["valid_pixels"]

    # K4 with the fused mark on the step's refined maps and grid
    pair, src = ops.build_pair_tables(sc.cam_from_world, sc.intrinsics, nbr, 0, V, H, W)
    sess = ops.FuseSession(torch.device("cuda"))
    grid = ref.host_grid()
    xyz = torch.empty((V, H, W, 3), dtype=torch.float32, device="cuda")
    votes = torch.empty((V, H, W), dtype=torch.uint8, device="cuda")
    sup = torch.empty_like(votes)
    bbox = ops.new_bbox(torch.device("cuda"))
    thr = ref.vote_threshold

    def k4(support):
        return lambda: ops.backproject_filter(ref.refined, sc.normal, nbr, pair, src, 0, thr, fopt, bbox=bbox, xyz_out=xyz,
                                              votes_out=votes, mark=sess, support=support, support_out=sup)

    k4s = {"support_m2": k4((2, TAU)), "support_m2_reproj_1px": k4((2, TAU, 1.0))}
    times = {k: [] for k in k4s}
    for _ in range(3):  # warm-up of every shape
        for f in k4s.values():
            sess.begin_grid(grid)
            f()
    torch.cuda.synchronize()
    for _ in range(samples):
        for k, f in k4s.items():
            sess.begin_grid(grid)
            times[k].append(timed(f))
    peak, src_peak = hbm_peak()
    bpp = 29 + 4 * K
    med = {k: float(np.median(v)) for k, v in times.items()}
    out["k4_with_mark_ms"] = med
    out["k4_ratio_reproj_over_support"] = med["support_m2_reproj_1px"] / med["support_m2"]
    out["k4_spread_ms"] = {k: [float(np.min(v)), float(np.max(v))] for k, v in times.items()}
    out["roofline_frac"] = {k: bpp * n_valid / (ms * 1e-3) / 1e9 / peak for k, ms in med.items()}
    out["roofline"] = {"algorithmic_bytes_per_pixel": bpp, "peak_gbs": peak, "peak_source": src_peak, "pixels": n_valid}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=15)
    ap.add_argument("--arm", choices=("support", "reproj"), default="support")
    ap.add_argument("--out", default=None, help="default: profiles/r09_support.json, or profiles/r10_support_reproj.json")
    args = ap.parse_args()
    if args.out is None:
        args.out = "profiles/r09_support.json" if args.arm == "support" else "profiles/r10_support_reproj.json"
    if not torch.cuda.is_available():
        raise SystemExit("support_bench needs a CUDA device")
    V, W, H, K, C, desc = WORKLOADS["cfg2"]
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=C, seed=0), device="cuda")
    nbr = torch.from_numpy(nearest_views_table(sc.cam_from_world.cpu().numpy(), K).astype(np.int32)).cuda()
    fn = line if args.arm == "support" else reproj_line
    res = {"card": card(), "workload": desc, "support_tau": TAU, "samples": args.samples,
           "lines": [fn(sc, nbr, m, args.samples) for m in ("nearest", "bilinear")]}
    res["card_after"] = card()
    print(json.dumps(res))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
