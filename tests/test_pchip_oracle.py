"""The FastPCHIP restatement (oracle/restatement_pchip.py) against the reference's own outputs: the committed
golden cases (tests/golden/ref_pchip_cases.npz, produced by oracle/make_golden.py from the unmodified
reference module)."""

import numpy as np
import pytest

from oracle import restatement_pchip as P
from oracle.restatement import kmatrix

CASES = {
    "default": dict(kw={}, mask=True, rgb=False, normal=True),
    "mask_none_no_normal": dict(kw={}, mask=False, rgb=False, normal=False),
    "image_edges": dict(kw=dict(use_image_edges=True, image_edge_threshold=12.0), mask=True, rgb=True, normal=True),
    "not_robust_tight": dict(kw=dict(robust=False, edge_threshold=0.02, edge_margin=5), mask=True, rgb=False, normal=True),
    "too_few": dict(kw=dict(min_correspondences=100000), mask=True, rgb=False, normal=True),
    "too_few_after_outliers": dict(kw=dict(outlier_threshold=1e-9, min_correspondences=50), mask=True, rgb=False, normal=True),
}


def case_args(g, name, v):
    sp = CASES[name]
    lo, hi = int(g["sparse_offsets"][v]), int(g["sparse_offsets"][v + 1])
    return dict(depth_map=g["mono_depth"][v].copy(), normal_map=g["normal"][v] if sp["normal"] else None,
                points3D=g["sparse_xyz"][lo:hi], cam_from_world=g["cam_from_world"][v], K=kmatrix(g["intrinsics"][v]),
                mask=g["mask"][v] if sp["mask"] else None, rgb_image=g["rgb"][v] if sp["rgb"] else None), sp["kw"]


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_matches_golden(golden_dir, name):
    g = np.load(golden_dir / "ref_pchip_cases.npz")
    for v in range(2):
        args, kw = case_args(g, name, v)
        out = P.refine_depth(cfg=P.PchipConfig(**kw), **args)
        assert np.array_equal(np.asarray(out["refined_depth"], np.float32), g[f"{name}/{v}/refined"])
        assert out["scale"] == float(g[f"{name}/{v}/scale"]) and out["num_iterations"] == int(g[f"{name}/{v}/iters"])
    # the cases really exercise what their names say
    it = int(g[f"{name}/0/iters"])
    assert it == (0 if name.startswith("too_few") else 1)
    if name == "too_few_after_outliers":
        assert float(g[f"{name}/0/scale"]) != 1.0


def test_restatement_matches_reference_module(golden_dir):
    """The restatement's output as it is returned (no cast), against the reference module's output."""
    g = np.load(golden_dir / "ref_pchip_cases.npz")
    for name in ("default", "image_edges"):
        args, kw = case_args(g, name, 1)
        mine = P.refine_depth(cfg=P.PchipConfig(**kw), **args)
        assert np.array_equal(g[f"{name}/1/refined"], mine["refined_depth"]) and float(g[f"{name}/1/scale"]) == mine["scale"]
