"""The multi-view support count and keep rule of K4 (ddn_backproject_filter_support*) against the host restatement in
tests/support_oracle.py, and the keep invariant through every layer: keep_mask(), the fused mark (counts[0]), dense,
hashed and host-grid fusion, the sharded densifier and pipeline.main.  Bars as in tests/parity.py: bit for bit outside
the tie bands, whose share is asserted small."""

import os

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import all_views_table, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import parity
import support_oracle as S
from test_gpu_vote_space import _cuda, _points, _refined

pytestmark = pytest.mark.gpu

TAU = 0.01


def _filter(refined, normal, poses, intr, nbr, thr, support=None, mark=None, **fopts):
    from depthdensifier_b200 import ops

    V, H, W = refined.shape
    d_nbr = _cuda(nbr.astype(np.int32))
    pair, src = ops.build_pair_tables(_cuda(poses), _cuda(intr), d_nbr, 0, V, H, W)
    bbox = ops.new_bbox(d_nbr.device)
    out = ops.backproject_filter(_cuda(refined), _cuda(normal), d_nbr, pair, src, 0, thr, ops.FilterOptions(**fopts), bbox=bbox,
                                 mark=mark, **({} if support is None else {"support": support}))
    torch.cuda.synchronize()
    return [o.cpu().numpy() for o in out] + [bbox.cpu().numpy()]


def _oracle_kw(fopts):
    kw = dict(sample_mode=fopts.get("sample_mode", "nearest"))
    if fopts.get("two_sided_tau", 0.0) > 0:
        kw["two_sided_tau"] = fopts["two_sided_tau"]
    return kw


def _check(sc, refined, nbr, m, thr=2, max_tie=0.01, tau=TAU, **fopts):
    """Support bytes and keep of K4 against the oracle; returns the oracle's (support, ties) and the device's votes."""
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    stride = fopts.get("stride", 1)
    xyz, votes, sup, _ = _filter(refined, normal, poses, intr, nbr, thr, support=(m, tau), **fopts)
    valid = refined[:, ::stride, ::stride] > 0
    assert np.array_equal(votes != 255, valid) and np.array_equal(sup != 255, valid)
    pts, nrm, src = _points(refined, normal, poses, intr, range(sc.n_views), stride)
    ref_s, sties, pair_frac = S.support_with_ties(pts, src, refined, poses, intr, nbr, tau, fopts.get("sample_mode", "nearest"))
    ref_v, vties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr, **_oracle_kw(fopts))
    clean = sties == 0
    got_s = sup[valid].astype(np.int64)
    bad = clean & (got_s != np.minimum(ref_s, 254))
    assert not bad.any(), f"{bad.sum()} of {clean.sum()} tie-free support counts differ"
    assert (np.abs(got_s - np.minimum(ref_s, 254)) <= sties).all()
    assert pair_frac <= max_tie, f"support tie fraction {pair_frac:.4f} of the (point, entry) pairs"
    both = clean & (vties == 0)
    keep = votes[valid] < min(thr, 254)
    assert np.array_equal(keep[both], S.keep(ref_v, ref_s, thr, m)[both])
    assert ref_s.max() >= 1 and (ref_s < ref_s.max()).any()
    return ref_s, sties, votes[valid]


@pytest.fixture(scope="module")
def scene48():
    sc = make_scene(SceneConfig(n_views=48, width=96, height=72, n_sparse=300, seed=5))
    return sc, _refined(sc)


@pytest.mark.parametrize("fopts", [
    dict(stride=1, pixel_layout=0),
    dict(stride=3, pixel_layout=1),
    dict(two_sided_tau=0.05),
    dict(sample_mode="bilinear", pixel_layout=1),
    dict(sample_mode="bilinear", two_sided_tau=0.05, stride=3, pixel_layout=0),
], ids=["nearest-s1-L0", "nearest-s3-L1", "nearest-two-sided", "bilinear-L1", "bilinear-two-sided-s3"])
@pytest.mark.parametrize("table", ["knn4", "knn40", "all48"])
def test_support_matches_oracle(lib_built, scene48, fopts, table):
    """K = 4, K = 40 of 48 (two neighbour blocks), and K = V = 48 with the own view in the table (never counted)."""
    sc, refined = scene48
    poses = sc.cam_from_world.numpy()
    nbr = {"knn4": lambda: nearest_views_table(poses, 4), "knn40": lambda: nearest_views_table(poses, 40),
           "all48": lambda: all_views_table(sc.n_views)}[table]()
    ref_s, _, _ = _check(sc, refined, nbr, 2, **fopts)
    if table != "knn4":  # the second block of 32 entries supports points too
        assert ref_s.max() > 4


def test_support_saturates_at_254(lib_built):
    """K = V = 300: counts past the u8 saturation (tau = 1: every in-bounds neighbour with a depth of at least half the
    point's supports it)."""
    sc = make_scene(SceneConfig(n_views=300, width=24, height=18, n_sparse=40, seed=3))
    refined = _refined(sc)
    ref_s, _, _ = _check(sc, refined, all_views_table(300), 260, thr=1000, tau=1.0)
    assert ref_s.max() > 254


def test_support_ragged(lib_built):
    """A mixed-size scene through ddn_backproject_filter_support_ragged against the per-view oracle."""
    from depthdensifier_b200 import ops

    sizes = [(48, 64), (40, 56), (64, 48), (52, 70), (48, 64), (36, 50)]
    scs = [make_scene(SceneConfig(n_views=6, width=w, height=h, n_sparse=300, seed=8)) for h, w in sizes]
    base = scs[0]
    poses, intr = base.cam_from_world.numpy(), base.intrinsics.numpy().copy()
    refined, normals = [], []
    for v, (h, w) in enumerate(sizes):
        r = _refined(scs[v])[v]
        refined.append(r)
        normals.append(scs[v].normal.numpy()[v])
        intr[v] = scs[v].intrinsics.numpy()[v]
    nbr = nearest_views_table(poses, 3)
    for stride in (1, 2):
        lay = ops.ViewLayout.from_shapes(sizes, stride)
        d_nbr = _cuda(nbr.astype(np.int32))
        pair, src = ops.build_pair_tables_ragged(lay, _cuda(poses), _cuda(intr), d_nbr)
        flat = lay.flatten([_cuda(r) for r in refined], torch.float32)
        nflat = lay.flatten([_cuda(n) for n in normals], torch.float32)
        xyz, votes, sup = ops.backproject_filter_ragged(lay, flat, nflat, pair, src, 2, ops.FilterOptions(stride=stride),
                                                        support=(1, TAU))
        sup = sup.cpu().numpy()
        pts, src_v = [], []
        for v in range(6):
            w_, py, px = R.backproject_view(refined[v], intr[v], poses[v], stride)
            pts.append(w_), src_v.append(np.full(len(w_), v))
        pts, src_v = np.concatenate(pts), np.concatenate(src_v)
        valid = sup != 255
        assert valid.sum() == len(pts)
        ref_s, ties, frac = S.support_with_ties(pts, src_v, refined, poses, intr, nbr, TAU)
        clean = ties == 0
        assert np.array_equal(sup[valid][clean], np.minimum(ref_s, 254)[clean]) and frac < 0.01
        assert ref_s.max() >= 2


@pytest.mark.parametrize("fopts", [dict(), dict(sample_mode="bilinear", stride=3, pixel_layout=1), dict(two_sided_tau=0.05)])
def test_min_support_zero_is_the_plain_kernel(lib_built, scene48, fopts):
    """m = 0, thr <= 254: votes, xyz, bbox and the fused mark equal ddn_backproject_filter's byte for byte."""
    from depthdensifier_b200 import ops

    sc, refined = scene48
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    nbr = nearest_views_table(poses, 6)
    outs = []
    for support in (None, (0, TAU)):
        sess = ops.FuseSession(torch.device("cuda"))
        sess.begin_grid(ops.make_grid(np.array([-20.0] * 3), np.array([20.0] * 3), 0.05))
        r = _filter(refined, normal, poses, intr, nbr, 3, support=support, mark=sess, **fopts)
        outs.append((r[0], r[1], r[-1], sess.units.cpu().numpy().copy(), sess.counts.cpu().numpy().copy()))
    for a, b in zip(*outs):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _engine_scene(dome=False):
    kw = dict(n_views=6, width=203, height=131, n_sparse=700, seed=9)
    if dome:
        kw["dome_radius"] = 150.0  # the grid exceeds the occupancy bitmap: hashed fusion
    return make_scene(SceneConfig(**kw))


def _engine_inputs(sc, nbr):
    return (sc.mono_depth.cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.cam_from_world.cuda(), sc.intrinsics.cuda(),
            sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), torch.from_numpy(nbr.astype(np.int32)).cuda())


@pytest.mark.parametrize("dome", [False, True], ids=["dense", "hashed"])
def test_keep_invariant_through_fusion(lib_built, dome):
    """At thr in {1, 5, 254, 255, 1000} x m in {0, 1, 2, K}: keep_mask() is the oracle's keep away from ties, counts[0]
    is its size, and the step's voxels (dense or hashed) and host-grid voxel_fuse are the oracle's voxel_fuse of the
    kept points."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = _engine_scene(dome)
    K = 5
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, K)
    voxel = 0.02
    inputs = _engine_inputs(sc, nbr)
    seen_status = set()
    for thr in (1, 5, 254, 255, 1000):
        for m in (0, 1, 2, K):
            eng = DensifyEngine(DensifyConfig(voxel=voxel, vote_threshold=thr, min_support=m, support_tau=TAU), device="cuda")
            res = eng.run(*inputs)
            seen_status.add(res.session.grid_state().status)
            refined = res.refined.cpu().numpy()
            valid = refined > 0
            keep = res.keep_mask().cpu().numpy()
            assert int(res.counts[0]) == int(keep.sum())
            # the oracle's keep on the device's refined maps
            pts, nrm, src = _points(refined, sc.normal.numpy(), poses, intr, range(sc.n_views))
            ref_v, vties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr)
            ref_s, sties, frac = S.support_with_ties(pts, src, refined, poses, intr, nbr, TAU)
            clean = (vties == 0) & (sties == 0)
            assert frac < 0.01 and clean.mean() > 0.8
            ok = S.keep(ref_v, ref_s, min(thr, 255), m)
            assert np.array_equal(keep[valid][clean], ok[clean]), (thr, m)
            assert np.array_equal(res.support.cpu().numpy()[valid][clean], np.minimum(ref_s, 254)[clean])
            xyz = res.xyz.cpu().numpy()[valid][keep[valid]]
            rgb = res.rgb.cpu().numpy()[valid][keep[valid]]
            if len(xyz) == 0:
                assert res.check() == 0
                continue
            origin = np.array(list(res.host_grid().origin), np.float32)
            k_ref, m_ref, c_ref, n_ref = R.voxel_fuse(xyz, rgb, voxel, origin)
            res.check()
            assert np.array_equal(res.voxel_keys.cpu().numpy().view(np.uint64), k_ref)
            assert np.array_equal(res.voxel_count.cpu().numpy(), n_ref) and np.array_equal(res.voxel_rgb.cpu().numpy(), c_ref)
            assert np.abs(res.voxel_xyz.cpu().numpy() - m_ref).max() <= 1e-5 * max(1.0, np.abs(m_ref).max())
            k2, x2, c2, n2, cnt2 = ops.voxel_fuse(res.xyz.view(-1, 3), res.rgb.view(-1, 3), res.votes.view(-1),
                                                  res.fusion_threshold(), res.host_grid(), row_len=res.xyz.shape[2])
            assert np.array_equal(k2.cpu().numpy().view(np.uint64), k_ref) and np.array_equal(n2.cpu().numpy(), n_ref)
    assert seen_status == ({4} if dome else {0})


def test_support_drops_a_patch_behind_the_surface(lib_built):
    """A patch of view 0's refined depth pushed 10 % BEHIND the surface: no neighbour votes against it (it is not in
    front of any surface), but with m = 1 no neighbour supports it either, so it is dropped - by K4 and by the oracle."""
    sc = make_scene(SceneConfig(n_views=8, width=128, height=96, n_sparse=400, seed=21))
    refined = _refined(sc)
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    patch = np.zeros(refined.shape[1:], bool)
    patch[30:60, 40:80] = True
    patch &= refined[0] > 0
    refined[0][patch] *= np.float32(1.1)
    nbr = nearest_views_table(poses, 4)
    votes0 = _filter(refined, normal, poses, intr, nbr, 2)[1]
    _, votes1, sup1, _ = _filter(refined, normal, poses, intr, nbr, 2, support=(1, TAU))
    keep_default = votes0[0][patch] < 2
    keep_support = votes1[0][patch] < 2
    assert keep_default.mean() > 0.9 and keep_support.mean() < 0.1
    pts, nrm, src = _points(refined, normal, poses, intr, [0])
    py, px = np.nonzero(refined[0] > 0)
    in_patch = patch[py, px]
    ref_v = R.consistency_votes(pts, nrm, src, refined, poses, intr, nbr)
    ref_s = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=TAU)
    assert (ref_v[in_patch] < 2).mean() > 0.9 and (S.keep(ref_v, ref_s, 2, 1)[in_patch]).mean() < 0.1


def test_sharded_one_rank_equals_engine(lib_built):
    """ShardedDensifier at one rank, support mode: votes, support and voxels equal DensifyEngine's through run and
    run_host."""
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = _engine_scene()
    V, H, W = sc.mono_depth.shape
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    cfg = DensifyConfig(voxel=0.02, min_support=2, support_tau=TAU)
    ref = DensifyEngine(cfg, device="cuda").run(*_engine_inputs(sc, nbr))
    mv = ref.check()
    sd = ShardedDensifier(cfg, torch.device("cuda"), 0, 1, V, 0, V, sc.cam_from_world, sc.intrinsics, nbr, H, W)
    dev_in = (sc.mono_depth.cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda())
    res = sd.run(*dev_in)
    n = res.check()
    assert n == mv and torch.equal(res.votes, ref.votes) and torch.equal(res.support, ref.support)
    assert torch.equal(res.keep_mask(), ref.keep_mask()) and int(res.counts[0]) == int(ref.counts[0])
    for a, b in ((res.voxel_keys, ref.voxel_keys), (res.voxel_count, ref.voxel_count), (res.voxel_rgb, ref.voxel_rgb),
                 (res.voxel_xyz, ref.voxel_xyz)):
        assert torch.equal(a[:n], b[:n])
    host = sd.pin_host_inputs(sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets)
    out = sd.run_host(*host)
    assert np.array_equal(out["keys"].numpy(), ref.voxel_keys.cpu().numpy())
    assert np.array_equal(out["xyz"].numpy(), ref.voxel_xyz.cpu().numpy())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_torchrun_two_ranks_support(lib_built):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", str(root / "scripts" / "check_multi_gpu.py"), "--min-support", "2"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_pipeline_main_min_support(lib_built, golden_dir, tmp_path):
    """``--filtering.min-support 2`` on the golden synthetic model: the model's appended points are the step's kept
    points (keep_mask under the support rule), a subset of what the default vote keeps."""
    import tyro

    from depthdensifier_b200 import pipeline as P
    from depthdensifier_b200.colmap_io import Reconstruction
    from test_gpu_pipeline import _write_scene

    g = np.load(golden_dir / "ref_main_allviews.npz")
    _write_scene(tmp_path, g)
    outs = {}
    for args in ([], ["--filtering.min-support", "2", "--filtering.support-tau", "0.01"]):
        cfg = tyro.cli(P.ScriptConfig, args=args)
        cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images",
                                  output_model_dir=tmp_path / f"out{len(args)}", depth_dir=tmp_path / "depth")
        cfg.processing.downsample_density = 1
        cfg.refiner.adaptive_correspondences = False
        cfg.filtering.vote_threshold = int(g["vote_threshold"])
        outs[len(args)] = (cfg, P.main(cfg, return_candidates=True))
    cfg, out = outs[4]
    assert cfg.filtering.min_support == 2 and abs(cfg.filtering.support_tau - 0.01) < 1e-12
    assert outs[0][0].filtering.min_support is None
    base = outs[0][1]
    assert np.array_equal(out.candidates, base.candidates)
    assert np.array_equal(out.points, out.candidates[out.keep]) and len(out.points) == out.keep.sum()
    assert not (out.keep & ~base.keep).any() and 0 < out.keep.sum() < base.keep.sum()
    dx, _ = Reconstruction(tmp_path / "out4").dense_points()
    assert np.array_equal(dx, out.points)
