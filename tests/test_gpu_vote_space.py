"""The consistency vote (K4) across the configurations it accepts, against the float64 statement through the C ABI.

The other parity tests run K4 at ten neighbours or fewer.  These run the tables past one 32-neighbour block (K = V = 48,
K = 40 of 48), up to the 1024-neighbour limit (110 KB of pair tables in shared memory, vote counts past the u8
saturation at 254), in every sampling mode with the own view in the table, at non-default thresholds, with world-frame
normals, and through the ragged path.  Bars as in tests/parity.py: bit for bit outside the stated tie bands."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import all_views_table, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R
from oracle.restatement_masks import transform_normals

import parity

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _refined(sc):
    """Stage 1 of the oracle for every view (float32, unmasked pixels zeroed, scripts/test.py:194)."""
    poses, intr, off = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.sparse_offsets.numpy()
    out = np.zeros(tuple(sc.mono_depth.shape), np.float32)
    for v in range(sc.n_views):
        r = R.refine_view(sc.mono_depth[v].numpy().copy(), sc.sparse_xyz.numpy()[off[v]:off[v + 1]], poses[v], R.kmatrix(intr[v]),
                          sc.mask[v].numpy(), R.AlignConfig(adaptive_correspondences=False))
        out[v] = r["refined_depth"]
        out[v][~sc.mask[v].numpy()] = 0
    return out


def _points(refined, normal, poses, intr, views, stride=1):
    """Back-projected points of ``views`` in K4's output order, with their camera-frame normals and source views."""
    pts, nrm, src = [], [], []
    for v in views:
        w, py, px = R.backproject_view(refined[v], intr[v], poses[v], stride)
        pts.append(w), nrm.append(normal[v][py, px]), src.append(np.full(len(w), v, np.int32))
    return np.concatenate(pts), np.concatenate(nrm), np.concatenate(src)


def _run_filter(refined, normal, poses, intr, nbr, thr, **fopts):
    from depthdensifier_b200 import ops

    V, H, W = refined.shape
    d_nbr = _cuda(nbr.astype(np.int32))
    pair, src = ops.build_pair_tables(_cuda(poses), _cuda(intr), d_nbr, 0, V, H, W)
    xyz, votes = ops.backproject_filter(_cuda(refined), _cuda(normal), d_nbr, pair, src, 0, thr, ops.FilterOptions(**fopts))
    torch.cuda.synchronize()
    return xyz.cpu().numpy(), votes.cpu().numpy()


def _oracle_kw(fopts):
    kw = dict(sample_mode=fopts.get("sample_mode", "nearest"))
    if fopts.get("two_sided_tau", 0.0) > 0:
        kw["two_sided_tau"] = fopts["two_sided_tau"]
    if "depth_threshold" in fopts:
        kw["depth_threshold"] = fopts["depth_threshold"]
    if "grazing_cos" in fopts:
        kw["grazing"] = fopts["grazing_cos"]
    return kw


@pytest.fixture(scope="module")
def scene48():
    """48 views at 96x72 (262k points): 47 neighbours of other views, i.e. two blocks of 32, plus the own view."""
    sc = make_scene(SceneConfig(n_views=48, width=96, height=72, n_sparse=300, seed=5))
    return sc, _refined(sc)


def _compare(sc, refined, nbr, max_tie_fraction, **fopts):
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    stride = fopts.get("stride", 1)
    xyz, votes = _run_filter(refined, normal, poses, intr, nbr, 2, **fopts)
    valid = refined[:, ::stride, ::stride] > 0
    assert votes.shape == valid.shape and np.array_equal(votes != 255, valid)
    pts, nrm, src = _points(refined, normal, poses, intr, range(sc.n_views), stride)
    assert np.abs(xyz[valid] - pts).max() <= RTOL * max(1.0, np.abs(pts).max())
    kw = _oracle_kw(fopts)
    ref, nties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr, **kw)
    assert np.array_equal(ref, R.consistency_votes(pts, nrm, src, refined, poses, intr, nbr, **kw))
    assert ref.max() >= 1
    frac = parity.assert_votes_match(votes[valid], ref, nties, max_tie_fraction=max_tie_fraction)
    return pts, nrm, src, ref, frac


@pytest.mark.parametrize("fopts", [
    dict(stride=1, pixel_layout=0),
    dict(stride=3, pixel_layout=1),
    dict(two_sided_tau=0.05),
    dict(sample_mode="bilinear", pixel_layout=1),
    dict(sample_mode="bilinear", two_sided_tau=0.05, stride=3),
    dict(depth_threshold=0.85, grazing_cos=0.3),
    dict(grazing_cos=-2.0, pixel_layout=1),
], ids=["nearest-s1-L0", "nearest-s3-L1", "nearest-two-sided", "bilinear", "bilinear-two-sided-s3", "thr0.85-cos0.3",
        "grazing-open"])
def test_all_views_table_past_one_neighbour_block(lib_built, scene48, fopts):
    """K = V = 48, the reference's own table (pipeline.main's default): two hot blocks and the own view."""
    sc, refined = scene48
    nbr = all_views_table(sc.n_views)
    pts, nrm, src, ref, _ = _compare(sc, refined, nbr, 0.05, **fopts)
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    if fopts.get("sample_mode") == "bilinear":  # the own view never votes: pair_ties_bilinear marked no tie there
        assert parity.own_view_votes(pts, nrm, src, refined, poses, intr, **_oracle_kw(fopts)) == 0
    # entries 32.. of the views 0..31 (their second block) are the views 33..47, and they vote
    first = src < 32
    late = R.consistency_votes(pts[first], nrm[first], src[first], refined, poses, intr, nbr, view_ids=set(range(33, 48)),
                               **_oracle_kw(fopts))
    assert late.max() >= 1


def test_nearest_table_past_one_neighbour_block(lib_built, scene48):
    """K = 40 nearest views of 48: the hot entries span two blocks and there is no own view."""
    sc, refined = scene48
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 40)
    assert (nbr >= 0).all() and not (nbr == np.arange(sc.n_views)[:, None]).any()
    _compare(sc, refined, nbr, 0.05)


@pytest.mark.parametrize("sample_mode", ["nearest", "bilinear"])
@pytest.mark.parametrize("table", ["knn", "all"])
def test_normals_in_world(lib_built, sample_mode, table):
    """normals_in_world: the grazing gate takes transform_normals of the pixel's normal (rotated by R_src^T and divided
    by |n| + 1e-8).  The normals are scaled per pixel by a seeded factor in [0.5, 2], so the normalisation decides."""
    sc = make_scene(SceneConfig(n_views=8, width=131, height=77, n_sparse=400, seed=19))
    refined = _refined(sc)
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    V = sc.n_views
    nbr = all_views_table(V) if table == "all" else nearest_views_table(poses, 3)
    normal = sc.normal.numpy() * np.random.default_rng(19).uniform(0.5, 2.0, refined.shape)[..., None].astype(np.float32)
    fopts = dict(sample_mode=sample_mode, normals_in_world=True, grazing_cos=0.5)
    xyz, votes = _run_filter(refined, normal, poses, intr, nbr, 2, **fopts)
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    pts, nrm_cam, src = _points(refined, normal, poses, intr, range(V))
    nrm = np.empty_like(nrm_cam, dtype=np.float64)
    for v in range(V):
        sel = src == v
        nrm[sel] = transform_normals(nrm_cam[sel], poses[v], np.ones(int(sel.sum()), bool))
    kw = _oracle_kw(fopts)
    ref, nties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr, **kw)
    parity.assert_votes_match(votes[valid], ref, nties, max_tie_fraction=0.02 if sample_mode == "nearest" else 0.08)
    # the case is sensitive to the normalisation: the rotated but unnormalised normals vote differently
    unnormalised = np.concatenate([(nrm_cam[src == v] @ poses[v][:, :3]) for v in range(V)])
    assert not np.array_equal(ref, R.consistency_votes(pts, unnormalised, src, refined, poses, intr, nbr, **kw))
    assert ref.max() >= 1


@pytest.fixture(scope="module")
def scene1024():
    sc = make_scene(SceneConfig(n_views=1024, width=40, height=30, n_sparse=60, seed=7))
    return sc, _refined(sc)


SAMPLED_VIEWS = (0, 341, 682, 1023)


def test_1024_neighbours_and_vote_saturation(lib_built, scene1024):
    """K = V = 1024, the largest table K4 takes (110 KB of shared memory).  With 1024 chances per point almost half the
    points have a tie pair somewhere, so the bars are per point: exact where there is none, within the tie count
    otherwise, and the u8 count saturates at 254 wherever the statement is sure to reach it."""
    sc, refined = scene1024
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    V = sc.n_views
    nbr = all_views_table(V)
    xyz, votes = _run_filter(refined, normal, poses, intr, nbr, 1000)
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    pts, nrm, src = _points(refined, normal, poses, intr, SAMPLED_VIEWS)
    got = np.concatenate([votes[v][valid[v]] for v in SAMPLED_VIEWS]).astype(np.int64)
    assert np.abs(np.concatenate([xyz[v][valid[v]] for v in SAMPLED_VIEWS]) - pts).max() <= RTOL * max(1.0, np.abs(pts).max())
    ref, nties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr)
    assert ref.max() >= 255  # saturation is exercised
    sat = np.minimum(ref, 254)
    clean = nties == 0
    assert np.array_equal(got[clean], sat[clean]), f"{(got[clean] != sat[clean]).sum()} of {clean.sum()} tie-free points differ"
    assert (np.abs(got - sat) <= nties).all()
    assert (got[ref - nties >= 254] == 254).all()


def test_1024_views_threshold_above_the_saturation_keeps_and_fuses_every_point(lib_built, scene1024):
    """vote_threshold = 1000 with points of 255 votes or more: K4's occupancy mark, fusion and keep_mask() must agree on
    keeping every valid point (DESIGN.md §1), and the voxels are the oracle's fusion of exactly those points."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc, _ = scene1024
    V = sc.n_views
    voxel = 0.1  # views that cannot be aligned from 60 sparse points pass through unscaled: the box is ~90 m wide
    align = ops.AlignOptions(adaptive_correspondences=False)
    res = DensifyEngine(DensifyConfig(align=align, voxel=voxel, vote_threshold=1000)).run(
        sc.mono_depth.cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.cam_from_world.cuda(), sc.intrinsics.cuda(),
        sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), _cuda(all_views_table(V).astype(np.int32)))
    res.check()
    votes = res.votes.cpu().numpy()
    n_valid = int((votes != 255).sum())
    assert (votes == 254).any()  # points at the saturated count exist
    keep = res.keep_mask()
    assert int(res.counts[0]) == int(keep.sum()) == int(res.voxel_count.sum()) == n_valid > 0
    xyz, rgb = res.kept_points()
    origin = np.array(list(res.host_grid().origin), np.float32)
    k, m, c, n = R.voxel_fuse(xyz.cpu().numpy(), rgb.cpu().numpy(), voxel, origin)
    mv = res.check()
    assert mv == len(k)
    assert np.array_equal(res.voxel_keys[:mv].cpu().numpy().view(np.uint64), k)
    assert np.array_equal(res.voxel_count[:mv].cpu().numpy(), n) and np.array_equal(res.voxel_rgb[:mv].cpu().numpy(), c)
    assert np.abs(res.voxel_xyz[:mv].cpu().numpy() - m).max() <= RTOL * max(1.0, np.abs(m).max())


@pytest.mark.parametrize("sample_mode,tau", [("nearest", 0.0), ("bilinear", 0.05)])
def test_ragged_path_past_one_neighbour_block(lib_built, sample_mode, tau):
    """A uniform 40-view scene through run_views with K = V gives run's bits (the ragged K4 reads every neighbour's
    size from its table entry, in both blocks)."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = make_scene(SceneConfig(n_views=40, width=64, height=48, n_sparse=200, seed=29), "cuda")
    nbr = torch.from_numpy(all_views_table(sc.n_views).astype(np.int32)).cuda()
    align = ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True)
    eng = DensifyEngine(DensifyConfig(align=align, filter=ops.FilterOptions(sample_mode=sample_mode, two_sided_tau=tau),
                                      voxel=0.02))
    args = (sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    a = eng.run(sc.mono_depth, sc.normal, sc.mask, sc.rgb, *args)
    b = eng.run_views(list(sc.mono_depth), list(sc.normal), list(sc.mask), list(sc.rgb), *args)
    assert a.check() > 0
    assert torch.equal(a.refined.view(-1), b.refined)
    assert torch.equal(a.xyz.view(-1, 3), b.xyz) and torch.equal(a.votes.view(-1), b.votes)
    assert int(a.votes[a.votes != 255].max()) >= 1
    assert torch.equal(a.keep_mask().view(-1), b.keep_mask())
    for f in ("voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
