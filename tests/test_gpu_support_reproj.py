"""The forward-backward reprojection form of K4's support count (ddn_backproject_filter_support_reproj*) against the
explicit host restatement in tests/reproj_oracle.py, and the keep invariant through every layer.  Bars as in
tests/parity.py: bit for bit outside the tie bands, whose share is asserted small; every comparison also shows that
the pixel bound decides some (point, entry) pairs the depth test alone would count."""

import os

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import all_views_table, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import parity
import reproj_oracle as RO
import support_oracle as S
from test_gpu_support import _engine_inputs, _engine_scene, _filter
from test_gpu_vote_space import _cuda, _points, _refined

pytestmark = pytest.mark.gpu

TAU = 0.01


def _filter_tables(refined, normal, poses, intr, nbr, thr, support, **fopts):
    """K4 through ops.backproject_filter; returns (xyz, votes, support bytes, (pair_table, src_table)) on the host."""
    from depthdensifier_b200 import ops

    V, H, W = refined.shape
    d_nbr = _cuda(nbr.astype(np.int32))
    pair, src = ops.build_pair_tables(_cuda(poses), _cuda(intr), d_nbr, 0, V, H, W)
    xyz, votes, sup = ops.backproject_filter(_cuda(refined), _cuda(normal), d_nbr, pair, src, 0, thr, ops.FilterOptions(**fopts),
                                             support=support)
    torch.cuda.synchronize()
    return xyz.cpu().numpy(), votes.cpu().numpy(), sup.cpu().numpy(), (pair.cpu().numpy(), src.cpu().numpy())


def _check(sc, refined, nbr, m, rho, thr=2, tau=TAU, max_tie=0.01, **fopts):
    """Support bytes of K4's reprojection form against the oracle; returns the oracle's support counts."""
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    stride = fopts.get("stride", 1)
    _, votes, sup, tables = _filter_tables(refined, normal, poses, intr, nbr, thr, (m, tau, rho), **fopts)
    valid = refined[:, ::stride, ::stride] > 0
    assert np.array_equal(votes != 255, valid) and np.array_equal(sup != 255, valid)
    pts, _, src = _points(refined, normal, poses, intr, range(sc.n_views), stride)
    ref_s, ties, frac, decided = RO.reproj_support_with_ties(pts, src, refined, poses, intr, nbr, tau, rho,
                                                             fopts.get("sample_mode", "nearest"), tables=tables)
    clean = ties == 0
    got = sup[valid].astype(np.int64)
    bad = clean & (got != np.minimum(ref_s, 254))
    assert not bad.any(), f"{bad.sum()} of {clean.sum()} tie-free support counts differ"
    assert (np.abs(got - np.minimum(ref_s, 254)) <= ties).all()
    assert frac <= max_tie, f"tie fraction {frac:.4f} of the (point, entry) pairs"
    assert decided > 0, "the pixel bound decides no (point, entry) pair here"
    supported = valid.copy()
    supported[valid] = ref_s >= m
    unsupported = valid & ~supported
    clean_v = np.zeros_like(valid)
    clean_v[valid] = clean
    assert (votes[unsupported & clean_v] == 254).all()
    return ref_s


@pytest.fixture(scope="module")
def scene48():
    sc = make_scene(SceneConfig(n_views=48, width=96, height=72, n_sparse=300, seed=5))
    return sc, _refined(sc)


FOPTS = [
    dict(stride=1, pixel_layout=0),
    dict(stride=3, pixel_layout=1),
    dict(two_sided_tau=0.05),
    dict(sample_mode="bilinear", pixel_layout=1),
    dict(sample_mode="bilinear", two_sided_tau=0.05, stride=3, pixel_layout=0),
]
FOPT_IDS = ["nearest-s1-L0", "nearest-s3-L1", "nearest-two-sided", "bilinear-L1", "bilinear-two-sided-s3"]


@pytest.mark.parametrize("fopts", FOPTS, ids=FOPT_IDS)
@pytest.mark.parametrize("table", ["knn4", "knn40", "all48"])
def test_reproj_matches_oracle(lib_built, scene48, fopts, table):
    """K = 4 (close neighbours: rho = 0.1 px), K = 40 of 48 (two neighbour blocks) and K = V = 48 with the own view in
    the table (rho = 1 px)."""
    sc, refined = scene48
    poses = sc.cam_from_world.numpy()
    nbr = {"knn4": lambda: nearest_views_table(poses, 4), "knn40": lambda: nearest_views_table(poses, 40),
           "all48": lambda: all_views_table(sc.n_views)}[table]()
    ref_s = _check(sc, refined, nbr, 2, 0.1 if table == "knn4" else 1.0, **fopts)
    assert ref_s.max() >= 2 and (ref_s < ref_s.max()).any()


def test_reproj_saturates_at_254(lib_built):
    """K = V = 300, tau = 1, rho = 20 px: counts past the u8 saturation, and the pixel bound still decides pairs."""
    sc = make_scene(SceneConfig(n_views=300, width=24, height=18, n_sparse=40, seed=3))
    ref_s = _check(sc, _refined(sc), all_views_table(300), 260, 20.0, thr=1000, tau=1.0)
    assert ref_s.max() > 254


def test_reproj_ragged(lib_built):
    """A mixed-size scene through ddn_backproject_filter_support_reproj_ragged against the oracle."""
    from depthdensifier_b200 import ops

    sizes = [(48, 64), (40, 56), (64, 48), (52, 70), (48, 64), (36, 50)]
    scs = [make_scene(SceneConfig(n_views=6, width=w, height=h, n_sparse=300, seed=8)) for h, w in sizes]
    poses, intr = scs[0].cam_from_world.numpy(), scs[0].intrinsics.numpy().copy()
    refined, normals = [], []
    for v in range(6):
        refined.append(_refined(scs[v])[v])
        normals.append(scs[v].normal.numpy()[v])
        intr[v] = scs[v].intrinsics.numpy()[v]
    nbr = nearest_views_table(poses, 3)
    for stride, rho in ((1, 0.1), (2, 0.2)):
        lay = ops.ViewLayout.from_shapes(sizes, stride)
        d_nbr = _cuda(nbr.astype(np.int32))
        pair, src = ops.build_pair_tables_ragged(lay, _cuda(poses), _cuda(intr), d_nbr)
        flat = lay.flatten([_cuda(r) for r in refined], torch.float32)
        nflat = lay.flatten([_cuda(n) for n in normals], torch.float32)
        _, _, sup = ops.backproject_filter_ragged(lay, flat, nflat, pair, src, 2, ops.FilterOptions(stride=stride),
                                                  support=(1, TAU, rho))
        sup = sup.cpu().numpy()
        pts, src_v = [], []
        for v in range(6):
            w_, _, _ = R.backproject_view(refined[v], intr[v], poses[v], stride)
            pts.append(w_), src_v.append(np.full(len(w_), v))
        pts, src_v = np.concatenate(pts), np.concatenate(src_v)
        valid = sup != 255
        assert valid.sum() == len(pts)
        ref_s, ties, frac, decided = RO.reproj_support_with_ties(pts, src_v, refined, poses, intr, nbr, TAU, rho,
                                                                 tables=(pair.cpu().numpy(), src.cpu().numpy()))
        clean = ties == 0
        assert np.array_equal(sup[valid][clean], np.minimum(ref_s, 254)[clean]) and frac < 0.01
        assert ref_s.max() >= 2 and decided > 0


@pytest.mark.parametrize("fopts", [dict(), dict(sample_mode="bilinear", stride=3, pixel_layout=1), dict(two_sided_tau=0.05),
                                   dict(stride=2, pixel_layout=1)])
def test_huge_rho_is_the_support_kernel(lib_built, scene48, fopts):
    """rho = 1e30: votes, support, xyz, bbox and the fused mark equal ddn_backproject_filter_support's byte for byte."""
    from depthdensifier_b200 import ops

    sc, refined = scene48
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    nbr = nearest_views_table(poses, 40)
    outs = []
    for support in ((2, TAU), (2, TAU, 1e30)):
        sess = ops.FuseSession(torch.device("cuda"))
        sess.begin_grid(ops.make_grid(np.array([-20.0] * 3), np.array([20.0] * 3), 0.05))
        r = _filter(refined, normal, poses, intr, nbr, 3, support=support, mark=sess, **fopts)
        outs.append((r[0], r[1], r[2], r[-1], sess.units.cpu().numpy().copy(), sess.counts.cpu().numpy().copy()))
    for a, b in zip(*outs):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))


@pytest.mark.parametrize("fopts", [dict(), dict(sample_mode="bilinear"), dict(two_sided_tau=0.05, stride=2, pixel_layout=1)])
def test_reproj_rig_in_closed_form(lib_built, fopts):
    """The translated-plane rig of tests/test_reproj_oracle.py on the device: view 1 returns 0.0274 px from where the
    round trip started, view 2 0.1078 px, so which entries support each point is known at every rho."""
    from test_reproj_oracle import ERR1, ERR2
    from test_support_oracle import W, plane_scene

    refined, poses, intr, pts, px = plane_scene()
    stride = fopts.get("stride", 1)
    normal = np.zeros(refined.shape + (3,), np.float32)
    normal[..., 2] = -1
    nbr = np.array([[1, 2], [0, 2], [0, 1]], np.int32)
    ys, xs = np.mgrid[0:refined.shape[1]:stride, 0:refined.shape[2]:stride]
    in1 = (xs >= 6).astype(np.int64)
    in2 = (xs <= W - 6).astype(np.int64)
    for rho, want in ((0.5 * ERR1, 0 * in1), (0.5 * (ERR1 + ERR2), in1), (2 * ERR2, in1 + in2)):
        _, votes, sup, _ = _filter_tables(refined, normal, poses, intr, nbr, 3, (1, 0.03, rho), **fopts)
        rows = ys[:, 0] > 0  # row 0 lies on the v = 0 border band
        assert np.array_equal(sup[0][rows], want[rows]), rho
        assert np.array_equal(votes[0][rows] == 254, want[rows] == 0)


def test_bad_rho_is_rejected(lib_built, scene48):
    """rho <= 0, inf and NaN never reach the device (the C entry points' own checks: tests/test_support_reproj_args.py)."""
    sc, refined = scene48
    poses, intr, normal = sc.cam_from_world.numpy(), sc.intrinsics.numpy(), sc.normal.numpy()
    nbr = nearest_views_table(poses, 4)
    for rho in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError):
            _filter(refined, normal, poses, intr, nbr, 2, support=(1, TAU, rho))


@pytest.mark.parametrize("dome", [False, True], ids=["dense", "hashed"])
def test_keep_invariant_through_fusion(lib_built, dome):
    """support_reproj_px = 1 at a few (thr, m): keep_mask() is the oracle's keep away from ties, counts[0] is its
    size, and the step's voxels (dense or hashed) and host-grid voxel_fuse are the oracle's voxel_fuse of the kept
    points."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = _engine_scene(dome)
    K = 5
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, K)
    voxel = 0.02
    inputs = _engine_inputs(sc, nbr)
    seen_status = set()
    for thr, m in ((1, 0), (5, 1), (254, 2), (1000, K)):
        eng = DensifyEngine(DensifyConfig(voxel=voxel, vote_threshold=thr, min_support=m, support_tau=TAU, support_reproj_px=1.0),
                            device="cuda")
        res = eng.run(*inputs)
        seen_status.add(res.session.grid_state().status)
        refined = res.refined.cpu().numpy()
        valid = refined > 0
        keep = res.keep_mask().cpu().numpy()
        assert int(res.counts[0]) == int(keep.sum())
        pts, nrm, src = _points(refined, sc.normal.numpy(), poses, intr, range(sc.n_views))
        ref_v, vties = parity.votes_with_ties(pts, nrm, src, refined, poses, intr, nbr)
        ref_s, sties, frac, _ = RO.reproj_support_with_ties(pts, src, refined, poses, intr, nbr, TAU, 1.0)
        clean = (vties == 0) & (sties == 0)
        assert frac < 0.01 and clean.mean() > 0.8
        assert np.array_equal(keep[valid][clean], S.keep(ref_v, ref_s, min(thr, 255), m)[clean]), (thr, m)
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


def test_sharded_one_rank_equals_engine(lib_built):
    """ShardedDensifier at one rank with the reprojection test: votes, support and voxels equal DensifyEngine's
    through run and run_host."""
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = _engine_scene()
    V, H, W = sc.mono_depth.shape
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    cfg = DensifyConfig(voxel=0.02, min_support=2, support_tau=TAU, support_reproj_px=0.5)
    plain = DensifyEngine(DensifyConfig(voxel=0.02, min_support=2, support_tau=TAU), device="cuda").run(*_engine_inputs(sc, nbr))
    ref = DensifyEngine(cfg, device="cuda").run(*_engine_inputs(sc, nbr))
    mv = ref.check()
    assert int(ref.counts[0]) <= int(plain.counts[0]) and (ref.support <= plain.support).all()
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
def test_torchrun_two_ranks_support_reproj(lib_built):
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", str(root / "scripts" / "check_multi_gpu.py"), "--min-support", "2", "--support-reproj-px", "1"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def test_pipeline_main_support_reproj(lib_built, golden_dir, tmp_path):
    """``--filtering.min-support 2 --filtering.support-reproj-px 1`` on the golden synthetic model: the appended points
    are the step's kept points, a subset of what the depth-only support test keeps."""
    import tyro

    from depthdensifier_b200 import pipeline as P
    from depthdensifier_b200.colmap_io import Reconstruction
    from test_gpu_pipeline import _write_scene

    g = np.load(golden_dir / "ref_main_allviews.npz")
    _write_scene(tmp_path, g)
    outs = {}
    for args in (["--filtering.min-support", "2"], ["--filtering.min-support", "2", "--filtering.support-reproj-px", "1"]):
        cfg = tyro.cli(P.ScriptConfig, args=args)
        cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images",
                                  output_model_dir=tmp_path / f"out{len(args)}", depth_dir=tmp_path / "depth")
        cfg.processing.downsample_density = 1
        cfg.refiner.adaptive_correspondences = False
        cfg.filtering.vote_threshold = int(g["vote_threshold"])
        outs[len(args)] = (cfg, P.main(cfg, return_candidates=True))
    cfg, out = outs[4]
    assert cfg.filtering.support_reproj_px == 1.0 and outs[2][0].filtering.support_reproj_px is None
    base = outs[2][1]
    assert np.array_equal(out.candidates, base.candidates)
    assert np.array_equal(out.points, out.candidates[out.keep]) and len(out.points) == out.keep.sum()
    assert not (out.keep & ~base.keep).any()
    dx, _ = Reconstruction(tmp_path / "out4").dense_points()
    assert np.array_equal(dx, out.points)
