"""The tie analysis of tests/parity.py must reproduce the float64 vote statement it brackets: whatever bands it adds,
the vote each helper returns is R.votes_against_view's, and the per-point sum is R.consistency_votes'.  Runs without a
GPU; the GPU tests then compare the kernel with these votes outside the ties."""

import numpy as np
import pytest

from depthdensifier_b200.neighbours import all_views_table, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import parity


@pytest.fixture(scope="module")
def scene():
    sc = make_scene(SceneConfig(n_views=6, width=131, height=77, n_sparse=400, seed=3))
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = all_views_table(6)
    out = R.densify(sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy(), sc.sparse_xyz.numpy(),
                    sc.sparse_offsets.numpy(), poses, intr, nbr, 3, align=R.AlignConfig(adaptive_correspondences=False))
    return out, poses, intr


VARIANTS = [
    ("nearest", None, {}),
    ("nearest", 0.05, {}),
    ("nearest", None, dict(depth_threshold=0.85, grazing=0.3)),
    ("nearest", 0.12, dict(depth_threshold=0.85, grazing=-2.0)),
    ("bilinear", None, {}),
    ("bilinear", 0.05, {}),
    ("bilinear", None, dict(depth_threshold=0.85, grazing=0.3)),
    ("bilinear", 0.12, dict(depth_threshold=0.85, grazing=-2.0)),
]


@pytest.mark.parametrize("table", ["all", "knn"])
@pytest.mark.parametrize("sample_mode,tau,kw", VARIANTS)
def test_tie_analysis_reproduces_the_statement(scene, table, sample_mode, tau, kw):
    out, poses, intr = scene
    refined, pts, nrm, src = out["refined"], out["points"], out["normals"], out["src_view"]
    V = refined.shape[0]
    nbr = all_views_table(V) if table == "all" else nearest_views_table(poses, 3)
    opts = dict(sample_mode=sample_mode, two_sided_tau=tau, **kw)
    fn = parity.pair_ties if sample_mode == "nearest" else parity.pair_ties_bilinear
    for t in range(V):  # each helper, view by view (own view included in the all-views table)
        sel = np.where((nbr[src] == t).any(1))[0]
        vote, tie = fn(pts[sel], nrm[sel], src[sel], t, refined[t], poses[t], intr[t], two_sided_tau=tau, **kw)
        ref = R.votes_against_view(pts[sel], nrm[sel], refined[t], poses[t], intr[t], **opts)
        assert np.array_equal(vote, ref), t
        assert tie.mean() < 0.05, (t, tie.mean())
    votes, nties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr, **opts)
    assert np.array_equal(votes, R.consistency_votes(pts, nrm, src, refined, poses, intr, nbr, **opts))
    assert votes.max() >= 1 and (nties == 0).mean() > 0.9
    if sample_mode == "bilinear" and table == "all":
        # the own view never votes in bilinear mode, so pair_ties_bilinear marks no own pair as a tie
        assert parity.own_view_votes(pts, nrm, src, refined, poses, intr, **opts) == 0


def test_two_sided_nearest_band(scene):
    """The two-sided nearest band brackets |z - D| = tau*D: moving tau onto a pair's own |z - D| / D makes it a tie."""
    out, poses, intr = scene
    refined, pts, nrm, src = out["refined"], out["points"], out["normals"], out["src_view"]
    t = 1
    sel = np.where(src != t)[0]
    _, det = R.votes_against_view(pts[sel], nrm[sel], refined[t], poses[t], intr[t], return_detail=True)
    D = det["D"].astype(np.float64)
    ok = det["inb"] & (D > 0)
    rel = np.abs(det["z"] - D)[ok] / D[ok]
    tau = float(np.median(rel))
    _, tie = parity.pair_ties(pts[sel], nrm[sel], src[sel], t, refined[t], poses[t], intr[t], two_sided_tau=tau)
    i = np.where(ok)[0][np.argmin(np.abs(rel - tau))]
    assert tie[i]
