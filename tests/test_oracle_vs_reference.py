"""Pins the oracle (oracle/restatement.py) to the reference: bit-identical to the reference's own outputs, stored
as golden vectors by oracle/make_golden.py."""

import numpy as np

from depthdensifier_b200.hashperm import hash_perm
from depthdensifier_b200.neighbours import all_views_table
from oracle import restatement as R
from oracle.make_golden import REFINER_FALLBACKS


def _densify_from_npz(g, **kw):
    V = g["mono_depth"].shape[0]
    return R.densify(
        g["mono_depth"], g["normal"], g["mask"], g["rgb"], g["sparse_xyz"], g["sparse_offsets"], g["cam_from_world"],
        g["intrinsics"], all_views_table(V), int(g["vote_threshold"]), depth_threshold=float(g["depth_threshold"]), **kw
    )


def test_golden_main_allviews(golden_dir):
    g = np.load(golden_dir / "ref_main_allviews.npz")
    out = _densify_from_npz(g, align=R.AlignConfig(adaptive_correspondences=False))
    assert np.array_equal(out["refined"], g["ref_refined"])
    assert np.array_equal(out["points"], g["ref_points"])
    assert np.array_equal(out["colors"], g["ref_colors"])
    assert np.array_equal(out["normals"], g["ref_normals"])
    assert np.array_equal(out["votes"], g["ref_votes"].astype(np.int64))
    assert np.array_equal(out["keep"], g["ref_keep"])
    assert np.array_equal(out["counts_per_view"], g["ref_counts_per_view"])
    # the reference's kept cloud is its points and colours at `keep` (make_golden.py checks that when it records the file)
    assert 0 < (~out["keep"]).sum() < len(out["keep"])  # the filter does real work on this scene


def test_golden_main_subsample_and_skipped_view(golden_dir):
    g = np.load(golden_dir / "ref_main_subsample.npz")
    out = _densify_from_npz(g, align=R.AlignConfig(), randperm=lambda n: hash_perm(n, 0))
    ids = g["ref_refined_view_ids"]
    assert list(out["active_views"]) == list(ids) and 2 not in ids  # view 2 has no sparse points
    assert np.array_equal(out["refined"][ids], g["ref_refined"])
    assert np.array_equal(out["points"], g["ref_points"])
    assert np.array_equal(out["colors"], g["ref_colors"])
    assert np.array_equal(out["votes"], g["ref_votes"].astype(np.int64))
    assert np.array_equal(out["keep"], g["ref_keep"])


def test_golden_refiner_cases(golden_dir):
    g = np.load(golden_dir / "ref_refiner_cases.npz")
    specs = {
        "default_hashperm": (R.AlignConfig(), True, True),
        "no_subsample": (R.AlignConfig(adaptive_correspondences=False), False, True),
        "skip_smoothing": (R.AlignConfig(adaptive_correspondences=False, skip_smoothing=True), False, True),
        "not_robust": (R.AlignConfig(adaptive_correspondences=False, robust=False), False, True),
        "mask_none": (R.AlignConfig(adaptive_correspondences=False), False, False),
        "too_few": (R.AlignConfig(min_correspondences=5000), False, True),
        "wide_margin": (R.AlignConfig(adaptive_correspondences=False, edge_margin=30, outlier_threshold=1.0), False, True),
    }
    for name, (cfg, perm, use_mask) in specs.items():
        for v in range(3):
            lo, hi = int(g["sparse_offsets"][v]), int(g["sparse_offsets"][v + 1])
            r = R.refine_view(
                g["mono_depth"][v].copy(), g["sparse_xyz"][lo:hi], g["cam_from_world"][v], R.kmatrix(g["intrinsics"][v]),
                g["mask"][v] if use_mask else None, cfg, randperm=(lambda n: hash_perm(n, 0)) if perm else None,
            )
            assert np.array_equal(np.asarray(r["refined_depth"], np.float32), g[f"{name}/{v}/refined"]), (name, v)
            assert r["num_correspondences"] == int(g[f"{name}/{v}/num"]), (name, v)
            assert r.get("outliers_removed", -1) == int(g[f"{name}/{v}/removed"]), (name, v)
            assert r["scale_factor"] == float(g[f"{name}/{v}/scale"]), (name, v)
    assert int(g["too_few/0/removed"]) == -1  # early-return dict has no outliers_removed key


def test_restatement_equals_unmodified_reference_main(golden_dir):
    g = np.load(golden_dir / "ref_main_seed11.npz")
    out = _densify_from_npz(g, randperm=lambda n: hash_perm(n, 5))
    assert np.array_equal(out["refined"], g["ref_refined"])
    assert np.array_equal(out["points"], g["ref_points"])
    assert np.array_equal(out["colors"], g["ref_colors"])
    assert np.array_equal(out["votes"], g["ref_votes"].astype(np.int64))
    assert np.array_equal(out["keep"], g["ref_keep"])


def test_restatement_equals_reference_refiner_stride_and_fallbacks(golden_dir):
    g = np.load(golden_dir / "ref_refiner_fallbacks.npz")
    for name, kw in REFINER_FALLBACKS.items():
        for v in range(2):
            lo, hi = int(g["sparse_offsets"][v]), int(g["sparse_offsets"][v + 1])
            args = (g["mono_depth"][v].copy(), g["sparse_xyz"][lo:hi], g["cam_from_world"][v], R.kmatrix(g["intrinsics"][v]), g["mask"][v])
            mine = R.refine_view(*args, R.AlignConfig(adaptive_correspondences=False, **kw))
            ref = {k.rsplit("/", 1)[1]: g[k] for k in g.files if k.startswith(f"{name}/{v}/")}
            assert np.array_equal(ref.pop("refined_depth"), np.asarray(mine["refined_depth"])), (name, v)
            assert {k: val.item() for k, val in ref.items()} == {k: mine[k] for k in mine if k != "refined_depth"}, (name, v)


def test_pwl_lookup_keeps_pair_order_of_repeated_knots():
    """Knots of equal x and different y, in shuffled pair order: a query at a repeated x takes the y of the repeat that
    comes first in pair order, a query just above it interpolates from the repeat that comes last (align_stats_kernel
    sorts by (x, pair index)).  Either answer changes when the two repeats trade places."""
    import torch

    rng = np.random.default_rng(3)
    reps = np.sort(rng.choice(np.arange(1, 99), 20, replace=False))
    x = np.concatenate([np.arange(100), reps]).astype(np.float32)
    order = rng.permutation(len(x))
    x = x[order]
    y = (rng.permutation(len(x)) * 2 + 1).astype(np.float32)  # distinct odd integers: every value below is exact
    queries, expected = [], []
    for r in reps:
        first, last = np.flatnonzero(x == r)  # pair order
        nxt = int(np.flatnonzero(x == r + 1)[0])  # searchsorted_left lands on the first knot of x = r + 1
        queries += [r, r + 0.5]
        expected += [y[first], y[last] + 0.5 * (y[nxt] - y[last])]
        assert y[first] != y[last]
    got = R.pwl_lookup(torch.tensor(queries, dtype=torch.float32), torch.from_numpy(x), torch.from_numpy(y))
    assert np.array_equal(got.numpy(), np.array(expected, np.float32))


def test_explicit_bilinear_matches_grid_sample():
    import torch
    import torch.nn.functional as F

    rng = np.random.default_rng(0)
    d = rng.uniform(0.5, 5, (37, 53)).astype(np.float32)
    u = rng.uniform(0, 52, 500).astype(np.float32)
    v = rng.uniform(0, 36, 500).astype(np.float32)
    grid = torch.stack([torch.from_numpy(u) / 52 * 2 - 1, torch.from_numpy(v) / 36 * 2 - 1], -1)[None, None]
    ref = F.grid_sample(torch.from_numpy(d)[None, None], grid, mode="bilinear", padding_mode="zeros", align_corners=True).squeeze().numpy()
    mine = R.bilinear_align_corners(d, u, v)
    assert (mine == ref).mean() > 0.999  # same operation order as ATen's CPU kernel
    np.testing.assert_allclose(mine, ref, rtol=3e-6, atol=1e-6)


def test_voxel_fuse_definition():
    rng = np.random.default_rng(1)
    xyz = rng.uniform(-1, 1, (5000, 3)).astype(np.float32)
    rgb = rng.integers(0, 256, (5000, 3)).astype(np.uint8)
    k, m, c, n = R.voxel_fuse(xyz, rgb, 0.05)
    assert (np.diff(k.astype(np.int64)) > 0).all() and n.sum() == 5000
    o = R.voxel_origin(xyz, 0.05)
    keys = R.voxel_keys(xyz, 0.05, o)
    j = int(np.argmax(n))
    sel = keys == k[j]
    np.testing.assert_allclose(m[j], xyz[sel].astype(np.float64).mean(0), rtol=1e-6)
    assert np.array_equal(c[j], np.floor(rgb[sel].astype(np.float64).mean(0) + 0.5).astype(np.uint8))
