"""TEST INFRASTRUCTURE ONLY - regenerate tests/golden/* from the reference's own code.

Needs a checkout of the original DepthDensifier (DDN_REFERENCE_ROOT):  python -m oracle.make_golden
The fixtures hold the inputs AND the outputs of the unmodified reference, so the tests pin the oracle
and the CUDA path to the reference on machines that do not have it.

ref_main_seed11.npz, ref_refiner_fallbacks.npz and ref_surface.json (sections 6-8) were first written
without the reference at hand: from the restatement and the package at the commit where the live
comparisons they stand in for passed against the reference (VERDICT.md, round 2: 52 passed, 0 skipped),
the surface without the fields and parameters the package marks as its own additions ("new", keyword-only,
FusionConfig).  Running this module against the reference rewrites them from the reference itself.
"""

from __future__ import annotations

import contextlib
import dataclasses
import inspect
import io
import json
import tempfile
from pathlib import Path

import numpy as np

from depthdensifier_b200.hashperm import hash_perm
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle.restatement import kmatrix
from oracle.run_reference import run_reference_main, run_reference_pchip, run_reference_refiner

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"

# (7) DepthRefiner.refine_depth without the random subsample: default, no smoothing, too few points, wide margin
REFINER_FALLBACKS = {"default": {}, "skip_smoothing": dict(skip_smoothing=True), "too_few": dict(min_correspondences=10_000),
                     "edge_margin_40": dict(edge_margin=40)}


def scene_arrays(sc):
    return dict(
        mono_depth=sc.mono_depth.numpy(), normal=sc.normal.numpy(), mask=sc.mask.numpy(), rgb=sc.rgb.numpy(),
        sparse_xyz=sc.sparse_xyz.numpy(), sparse_offsets=sc.sparse_offsets.numpy(),
        cam_from_world=sc.cam_from_world.numpy(), intrinsics=sc.intrinsics.numpy(),
    )


def main():
    GOLDEN.mkdir(parents=True, exist_ok=True)
    # (1) whole main(), all-views semantics (K = V), no random subsample
    sc = make_scene(SceneConfig(n_views=6, width=96, height=72, n_sparse=384, seed=0))
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ref = run_reference_main(sc, vote_threshold=2, adaptive_correspondences=False)
    # the cloud the reference adds to the model is its candidates at `keep`: checked here, so the file (< 1 MB) does
    # not carry that copy
    assert np.array_equal(ref["kept_points"], ref["points"][ref["keep"]])
    assert np.array_equal(ref["kept_colors"], ref["colors"][ref["keep"]])
    np.savez_compressed(
        GOLDEN / "ref_main_allviews.npz", vote_threshold=2, depth_threshold=0.7, **scene_arrays(sc),
        ref_refined=ref["refined"], ref_points=ref["points"], ref_colors=ref["colors"], ref_normals=ref["normals"],
        ref_votes=ref["votes"].astype(np.int16), ref_keep=ref["keep"], ref_counts_per_view=ref["counts_per_view"],
    )
    print("ref_main_allviews:", ref["points"].shape, "kept", int(ref["keep"].sum()), "vote hist", np.bincount(ref["votes"]))

    # (2) main() with the 500-subsample driven by the hash permutation and one view without sparse points
    sc2 = make_scene(SceneConfig(n_views=5, width=96, height=72, n_sparse=900, seed=7))
    off = sc2.sparse_offsets.numpy().copy()
    # drop the sparse points of view 2 (scripts/test.py:136-137 skips such views)
    lo, hi = int(off[2]), int(off[3])
    keep_rows = np.ones(off[-1], bool)
    keep_rows[lo:hi] = False
    import torch
    sc2.sparse_xyz = sc2.sparse_xyz[torch.from_numpy(keep_rows)]
    off[3:] -= hi - lo
    sc2.sparse_offsets = torch.from_numpy(off)
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ref2 = run_reference_main(sc2, vote_threshold=2, randperm=lambda n: hash_perm(n, 0))
    np.savez_compressed(
        GOLDEN / "ref_main_subsample.npz", vote_threshold=2, depth_threshold=0.7, **scene_arrays(sc2),
        ref_refined=ref2["refined"], ref_refined_view_ids=ref2["refined_view_ids"], ref_points=ref2["points"],
        ref_colors=ref2["colors"], ref_votes=ref2["votes"].astype(np.int16), ref_keep=ref2["keep"],
        ref_counts_per_view=ref2["counts_per_view"],
    )
    print("ref_main_subsample:", ref2["points"].shape, "kept", int(ref2["keep"].sum()), "views", ref2["refined_view_ids"])

    # (3) DepthRefiner.refine_depth cases
    sc3 = make_scene(SceneConfig(n_views=3, width=160, height=120, n_sparse=700, seed=3))
    a = scene_arrays(sc3)
    cases = {}
    specs = {
        "default_hashperm": dict(kw={}, perm=True, mask=True),
        "no_subsample": dict(kw=dict(adaptive_correspondences=False), perm=False, mask=True),
        "skip_smoothing": dict(kw=dict(adaptive_correspondences=False, skip_smoothing=True), perm=False, mask=True),
        "not_robust": dict(kw=dict(adaptive_correspondences=False, robust=False), perm=False, mask=True),
        "mask_none": dict(kw=dict(adaptive_correspondences=False), perm=False, mask=False),
        "too_few": dict(kw=dict(min_correspondences=5000), perm=False, mask=True),
        "wide_margin": dict(kw=dict(adaptive_correspondences=False, edge_margin=30, outlier_threshold=1.0), perm=False, mask=True),
    }
    for name, sp in specs.items():
        for v in range(3):
            lo, hi = int(a["sparse_offsets"][v]), int(a["sparse_offsets"][v + 1])
            r = run_reference_refiner(
                a["mono_depth"][v].copy(), a["sparse_xyz"][lo:hi], a["cam_from_world"][v], kmatrix(a["intrinsics"][v]),
                a["mask"][v] if sp["mask"] else None, randperm=(lambda n: hash_perm(n, 0)) if sp["perm"] else None, **sp["kw"],
            )
            cases[f"{name}/{v}/refined"] = np.asarray(r["refined_depth"], dtype=np.float32)
            cases[f"{name}/{v}/num"] = np.int64(r["num_correspondences"])
            cases[f"{name}/{v}/removed"] = np.int64(r.get("outliers_removed", -1))
            cases[f"{name}/{v}/scale"] = np.float64(r["scale_factor"])
    np.savez_compressed(GOLDEN / "ref_refiner_cases.npz", **a, **cases)
    print("ref_refiner_cases:", len(cases) // 4, "cases")

    # (4) FastPCHIPRefiner.refine_depth cases (fast_pchip_refiner.py:386-548)
    sc4 = make_scene(SceneConfig(n_views=2, width=176, height=128, n_sparse=900, seed=9))
    b = scene_arrays(sc4)
    pc = {}
    pspecs = {
        "default": dict(kw={}, mask=True, rgb=False, normal=True),
        "mask_none_no_normal": dict(kw={}, mask=False, rgb=False, normal=False),
        "image_edges": dict(kw=dict(use_image_edges=True, image_edge_threshold=12.0), mask=True, rgb=True, normal=True),
        "not_robust_tight": dict(kw=dict(robust=False, edge_threshold=0.02, edge_margin=5), mask=True, rgb=False, normal=True),
        "too_few": dict(kw=dict(min_correspondences=100000), mask=True, rgb=False, normal=True),
        "too_few_after_outliers": dict(kw=dict(outlier_threshold=1e-9, min_correspondences=50), mask=True, rgb=False, normal=True),
    }
    for name, sp in pspecs.items():
        for v in range(2):
            lo, hi = int(b["sparse_offsets"][v]), int(b["sparse_offsets"][v + 1])
            r = run_reference_pchip(
                b["mono_depth"][v].copy(), b["normal"][v] if sp["normal"] else None, b["sparse_xyz"][lo:hi], b["cam_from_world"][v],
                kmatrix(b["intrinsics"][v]), b["mask"][v] if sp["mask"] else None, rgb_image=b["rgb"][v] if sp["rgb"] else None, **sp["kw"])
            pc[f"{name}/{v}/refined"] = np.asarray(r["refined_depth"], dtype=np.float32)
            pc[f"{name}/{v}/scale"] = np.float64(r["scale"])
            pc[f"{name}/{v}/iters"] = np.int64(r["num_iterations"])
    np.savez_compressed(GOLDEN / "ref_pchip_cases.npz", **b, **pc)
    print("ref_pchip_cases:", len(pc) // 3, "cases")

    # (5) compute_depth_normal_gradient_mask (initilizer.py:236-328) on the same maps
    import importlib.util

    import torch
    from oracle.run_reference import REFERENCE_ROOT

    spec = importlib.util.spec_from_file_location("ddn_reference_init", REFERENCE_ROOT / "src" / "depthdensifier" / "initilizer.py")
    init = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(init)
    mc = {"mono_depth": b["mono_depth"], "normal": b["normal"]}
    for name, kw in {"default": {}, "tight": dict(depth_threshold=0.02, normal_threshold=0.1, edge_sigma=2.0),
                     "no_blur": dict(edge_sigma=0.0, depth_threshold=0.05)}.items():
        for v in range(2):
            for with_normal in (True, False):
                m = init.compute_depth_normal_gradient_mask(torch.from_numpy(b["mono_depth"][v]),
                                                            torch.from_numpy(b["normal"][v]) if with_normal else None, **kw)
                mc[f"{name}/{v}/{int(with_normal)}"] = m.numpy()
    np.savez_compressed(GOLDEN / "ref_mask_cases.npz", **mc)
    print("ref_mask_cases:", len(mc) - 2, "cases")

    main_seed11()
    refiner_fallbacks()
    reference_surface()


def main_seed11():
    """(6) main() with the 500-subsample driven by hash permutation 5, vote threshold 3 and depth ratio 0.8."""
    sc = make_scene(SceneConfig(n_views=5, width=112, height=80, n_sparse=600, seed=11))
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        ref = run_reference_main(sc, vote_threshold=3, depth_threshold=0.8, randperm=lambda n: hash_perm(n, 5))
    np.savez_compressed(
        GOLDEN / "ref_main_seed11.npz", vote_threshold=3, depth_threshold=0.8, **scene_arrays(sc), ref_refined=ref["refined"],
        ref_points=ref["points"], ref_colors=ref["colors"], ref_votes=ref["votes"].astype(np.int16), ref_keep=ref["keep"],
    )
    print("ref_main_seed11:", ref["points"].shape, "kept", int(ref["keep"].sum()))


def refiner_fallbacks():
    """(7) DepthRefiner.refine_depth: every key of the returned dict, for the REFINER_FALLBACKS cases."""
    a = scene_arrays(make_scene(SceneConfig(n_views=2, width=96, height=64, n_sparse=300, seed=5)))
    cases = {}
    for name, kw in REFINER_FALLBACKS.items():
        for v in range(2):
            lo, hi = int(a["sparse_offsets"][v]), int(a["sparse_offsets"][v + 1])
            r = run_reference_refiner(a["mono_depth"][v].copy(), a["sparse_xyz"][lo:hi], a["cam_from_world"][v],
                                      kmatrix(a["intrinsics"][v]), a["mask"][v], adaptive_correspondences=False, **kw)
            cases.update({f"{name}/{v}/{k}": np.asarray(val) for k, val in r.items()})
    np.savez_compressed(GOLDEN / "ref_refiner_fallbacks.npz", **a, **cases)
    print("ref_refiner_fallbacks:", len(REFINER_FALLBACKS) * 2, "cases")


def _defaults(dc) -> dict:
    """{field: repr(default)} of a dataclass; a required field or a default_factory reads 'None'."""
    return {f.name: repr(f.default if f.default is not dataclasses.MISSING else None) for f in dataclasses.fields(dc)}


def _params(fn) -> list:
    return [p for p in inspect.signature(fn).parameters if p != "self"]


def surface(refiner, script, pchip, gradient_mask, batch_config) -> dict:
    """The drop-in surface of one implementation: config fields with their defaults and the parameter lists of the
    entry points.  ``refiner``: module with RefinerConfig / DepthRefiner; ``script``: the pipeline module
    (scripts/test.py); ``pchip``: the fast_pchip_refiner module."""
    return {
        "RefinerConfig": _defaults(refiner.RefinerConfig),
        "DepthRefiner.__init__": _params(refiner.DepthRefiner.__init__),
        "DepthRefiner.refine_depth": _params(refiner.DepthRefiner.refine_depth)[:6],
        **{name: _defaults(getattr(script, name)) for name in ("PathsConfig", "MoGeConfig", "ProcessingConfig", "FilteringConfig")},
        "ScriptConfig": list(_defaults(script.ScriptConfig)),
        "project_points": _params(script.project_points),
        "unproject_points": _params(script.unproject_points),
        "main": _params(script.main)[:1],
        "FastPCHIPRefinerConfig": _defaults(pchip.FastPCHIPRefinerConfig),
        "FastPCHIPRefiner.__init__": _params(pchip.FastPCHIPRefiner.__init__),
        "FastPCHIPRefiner.refine_depth": _params(pchip.FastPCHIPRefiner.refine_depth),
        "refine_depth_from_colmap": _params(pchip.refine_depth_from_colmap),
        "compute_depth_normal_gradient_mask": [[p.name, repr(p.default)] for p in inspect.signature(gradient_mask).parameters.values()],
        "BatchConfig": [[f.name, f.default is dataclasses.MISSING and f.default_factory is dataclasses.MISSING]
                        for f in dataclasses.fields(batch_config)],
    }


def batch_output_dir(batch, tmp: Path) -> str:
    """Where ``batch.main`` (scripts/run_batch.py) sends the model of the first scan it densifies, relative to
    output_dir, over a root with one complete scan and one without sparse/0; densification itself is stubbed out."""
    (tmp / "root" / "scan_a" / "sparse" / "0").mkdir(parents=True)
    (tmp / "root" / "scan_a" / "images").mkdir()
    (tmp / "root" / "incomplete").mkdir()
    seen, densify = [], batch.densify_main
    batch.densify_main = lambda cfg: seen.append(Path(cfg.paths.output_model_dir))
    try:
        batch.main(batch.BatchConfig(root_dir=tmp / "root", output_dir=tmp / "out"))
    finally:
        batch.densify_main = densify
    return seen[0].relative_to(tmp / "out").as_posix()


def reference_surface():
    """(8) the reference's drop-in surface and batch output layout -> ref_surface.json."""
    import importlib.util
    import sys

    from oracle.run_reference import REFERENCE_ROOT, _import_reference_script, import_reference_pchip, import_reference_refiner

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    script = _import_reference_script()  # installs the stand-ins
    sys.modules["test"] = script  # scripts/run_batch.py imports the pipeline as `test`
    init = load("ddn_ref_init_sig", REFERENCE_ROOT / "src" / "depthdensifier" / "initilizer.py")
    batch = load("ddn_ref_run_batch", REFERENCE_ROOT / "scripts" / "run_batch.py")
    s = surface(import_reference_refiner(), script, import_reference_pchip(), init.compute_depth_normal_gradient_mask, batch.BatchConfig)
    with tempfile.TemporaryDirectory() as tmp:
        s["batch_output_model_dir"] = batch_output_dir(batch, Path(tmp))
    (GOLDEN / "ref_surface.json").write_text(json.dumps(s, indent=1) + "\n")
    print("ref_surface:", len(s), "entries")


if __name__ == "__main__":
    main()
