"""GPU tests of the hashed fusion path (include/ddn_b200.h: ddn_fuse_finish_hashed): voxel fusion for grids whose box
is too large for the session's dense occupancy bitmap.  Where both paths can run they must give the same bits; where
only the hashed one can, it must give the oracle's voxels."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import default_vote_threshold, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_mixed_scene, make_scene
from oracle import restatement as R

pytestmark = pytest.mark.gpu

DOME = dict(n_views=6, width=203, height=131, n_sparse=700, seed=9, dome_radius=150.0)  # box > 2^35 cells at 0.02
DOME_VOXEL = 0.02


def _cuda(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda().contiguous()


def _enc(f):
    i = f.astype(np.float32).view(np.int32)
    return np.where(i >= 0, i, i ^ np.int32(0x7FFFFFFF))


def _box(lo, hi):
    from depthdensifier_b200 import ops

    box = ops.new_bbox("cuda")
    box.copy_(torch.from_numpy(np.concatenate([_enc(np.asarray(lo)), _enc(np.asarray(hi))])))
    return box


def _assert_same_voxels(a, b, mv):
    for x, y in zip(a[:4], b[:4]):
        assert torch.equal(x[:mv], y[:mv])


def _assert_oracle_voxels(keys, xyz, rgb, cnt, kept_xyz, kept_rgb, voxel, origin):
    uk, mean, col, c = R.voxel_fuse(kept_xyz.astype(np.float32), kept_rgb, voxel, np.asarray(origin, np.float32))
    assert np.array_equal(keys.view(np.uint64), uk)
    assert np.array_equal(cnt, c) and np.array_equal(rgb, col)
    scale = max(1.0, float(np.abs(mean).max())) if len(mean) else 1.0
    assert len(mean) == 0 or np.abs(xyz - mean).max() <= 1e-5 * scale


def _clouds():
    rng = np.random.default_rng(5)
    out = {}
    n = 150000
    xyz = rng.normal(0, 0.7, (n, 3)).astype(np.float32)
    votes = rng.integers(0, 6, n).astype(np.uint8)
    votes[rng.random(n) < 0.05] = 255
    out["threshold_drops"] = (xyz, votes, 3, 0.02)
    out["empty"] = (np.zeros((0, 3), np.float32), np.zeros(0, np.uint8), 3, 0.02)
    out["all_dropped"] = (xyz[:5000], np.full(5000, 7, np.uint8), 3, 0.02)
    # one voxel holding 20000 points (625 warps of 32), next to a few scattered ones
    one = np.full((20000, 3), 0.013, np.float32) + rng.uniform(0, 0.0049, (20000, 3)).astype(np.float32)
    out["one_voxel"] = (np.concatenate([one, xyz[:300]]), np.zeros(20300, np.uint8), 1, 0.01)
    # nearly every point its own voxel (400000 keys in a 2^20-slot table, so probe sequences run into each other), and
    # dense clusters whose cells fill whole 64-slot brick blocks and spill into the next ones
    wide = np.concatenate([rng.uniform(-40, 40, (400000, 3)), rng.uniform(0, 0.4, (100000, 3))]).astype(np.float32)
    out["many_voxels"] = (wide, np.zeros(len(wide), np.uint8), 1, 0.05)
    return out


CLOUDS = _clouds()


@pytest.mark.parametrize("row_len", [0, 400])
@pytest.mark.parametrize("case", sorted(CLOUDS))
def test_hashed_equals_dense_and_oracle(lib_built, case, row_len):
    """Mode 1 on the session's own grid: the same keys, counts, colours, positions and counts[] as the dense finish,
    as ddn_voxel_fuse on the host copy of that grid, and as the oracle at the device origin."""
    from depthdensifier_b200 import _lib, ops

    xyz, votes, thr, voxel = CLOUDS[case]
    n = len(xyz)
    rgb = np.random.default_rng(n).integers(0, 256, (n, 3)).astype(np.uint8)
    d_xyz, d_rgb, d_votes = _cuda(xyz), _cuda(rgb), _cuda(votes)
    lo = xyz.min(0) - 0.013 if n else np.zeros(3, np.float32)
    hi = xyz.max(0) + 0.021 if n else np.ones(3, np.float32)
    sess = ops.FuseSession("cuda", max_cells=1 << 34)
    sess.begin([_box(lo, hi)], voxel)
    assert sess.grid_state().status == _lib.GRID_OK
    sess.mark_points(d_xyz, d_votes, thr)
    dense = [t.clone() for t in ops.fuse_finish(sess, d_xyz, d_rgb, d_votes, thr, row_len=row_len)]
    hf = ops.HashFuse("cuda", max(n, 1))
    hashed = ops.fuse_finish_hashed(sess, hf, d_xyz, d_rgb, d_votes, thr, row_len=row_len, mode=1)
    assert hf.ran()
    hf.check()
    n_pts, mv = hashed[4].cpu().tolist()
    assert [n_pts, mv] == dense[4].cpu().tolist()
    _assert_same_voxels(hashed, dense, mv)
    grid = sess.host_grid()
    host = ops.voxel_fuse(d_xyz, d_rgb, d_votes, thr, grid, row_len=row_len)
    assert host[4].cpu().tolist() == [n_pts, mv]
    _assert_same_voxels(hashed, host, mv)
    keep = votes < thr
    assert n_pts == int(keep.sum())
    _assert_oracle_voxels(*(t[:mv].cpu().numpy() for t in hashed[:4]), xyz[keep], rgb[keep], voxel, list(grid.origin))
    if case == "one_voxel":
        assert int(hashed[3][:mv].max()) >= 20000


def _scene_args(sc, nbr):
    return (sc.mono_depth.cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.cam_from_world.cuda(), sc.intrinsics.cuda(),
            sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), _cuda(nbr.astype(np.int32)))


def _engine(max_cells=None, voxel=0.02, **kw):
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    cfg = DensifyConfig(voxel=voxel, align=ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True), **kw)
    if max_cells is not None:
        cfg.max_grid_cells = max_cells
    return DensifyEngine(cfg)


def _status(res):
    return res.session.grid_state().status


def _voxels(res):
    return tuple(t.cpu().numpy() for t in (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.counts))


@pytest.mark.parametrize("dedup", [False, True])
@pytest.mark.parametrize("stride", [1, 3])
@pytest.mark.parametrize("form", ["run", "run_views"])
def test_engine_hashed_equals_dense(lib_built, form, stride, dedup):
    """The same scene through the dense path (default max_grid_cells) and the hashed one (1 << 16 cells): bit-identical
    voxels and counts, for run and run_views (a mixed-size scene); with dedup, the dense voxels minus the cells of the
    sparse cloud (merge_sparse(dedup=True))."""
    from depthdensifier_b200 import _lib, ops

    opts = dict(filter=ops.FilterOptions(stride=stride), dedup_sparse=dedup)
    if form == "run":
        sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
        nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
        call = lambda eng: eng.run(*_scene_args(sc, nbr))
    else:
        sc = make_mixed_scene(SceneConfig(n_sparse=400, seed=17), [(77, 131), (131, 77), (64, 96), (96, 64), (101, 127), (45, 63)])
        nbr = nearest_views_table(sc.cam_from_world.numpy(), 3)
        rest = (sc.cam_from_world.cuda(), sc.intrinsics.cuda(), sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), _cuda(nbr.astype(np.int32)))
        maps = [[m.cuda() for m in x] for x in (sc.mono_depth, sc.normal, sc.mask, sc.rgb)]
        call = lambda eng: eng.run_views(*maps, *rest)
    dense = call(_engine(**opts))
    hashed = call(_engine(max_cells=1 << 16, **opts))
    assert _status(dense) == _lib.GRID_OK and _status(hashed) == _lib.GRID_HASHED
    assert not dense.hash.ran() and hashed.hash.ran()
    a, b = _voxels(dense), _voxels(hashed)
    assert len(a[0]) > 1000
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    if dedup:
        plain = _voxels(call(_engine(max_cells=1 << 16, filter=ops.FilterOptions(stride=stride))))
        grid = hashed.host_grid()
        origin = np.array(list(grid.origin), np.float32)
        keys = plain[0].view(np.uint64)
        sparse = sc.sparse_xyz.numpy()
        merged, _ = R.merge_sparse(sparse, np.zeros((len(sparse), 3), np.uint8), plain[1], plain[2], dense_keys=keys, voxel=0.02,
                                   origin=origin, dedup=True)
        s32 = sparse.astype(np.float32)
        k3 = np.floor((s32 - origin) / np.float32(0.02)).astype(np.int64)
        sk = (k3[:, 0] | (k3[:, 1] << 21) | (k3[:, 2] << 42)).astype(np.uint64)
        keep = ~np.isin(keys, sk)
        assert 0 < keep.sum() < len(keys)
        assert np.array_equal(b[0].view(np.uint64), keys[keep]) and np.array_equal(b[1], plain[1][keep])
        assert np.array_equal(b[2], plain[2][keep]) and np.array_equal(b[3], plain[3][keep])
        assert np.array_equal(merged[len(sparse):], plain[1][keep].astype(np.float64))
        assert b[4][0] == plain[4][0]  # the points of removed cells still count, as on the dense path


def _kept(res):
    xyz, rgb = res.kept_points()
    return xyz.cpu().numpy(), rgb.cpu().numpy()


def test_unbounded_dome_scene(lib_built):
    """A scene with distant background: the box of what the views see exceeds 2^35 cells (tests/test_hashed_fuse_host.py
    checks it on the host), the dense path cannot hold it at any session size, the step completes through the hash
    table with the oracle's voxels of the kept points at the device origin."""
    from depthdensifier_b200 import _lib

    sc = make_scene(SceneConfig(**DOME))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    res = _engine(voxel=DOME_VOXEL).run(*_scene_args(sc, nbr))
    assert _status(res) == _lib.GRID_HASHED
    st = res.session.grid_state()
    assert st.cells > (1 << 35)
    kx, krgb = _kept(res)
    assert int(res.counts[0]) == len(kx)
    grid = res.host_grid()
    _assert_oracle_voxels(*_voxels(res)[:4], kx, krgb, DOME_VOXEL, list(grid.origin))


def test_one_outlier_depth_no_longer_fails(lib_built):
    """Every view passes its depth through unaligned, and one pixel has 10^4 x its depth: the box becomes far too large
    for the session, and the step still completes with the oracle's voxels."""
    from depthdensifier_b200 import _lib, ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    sc.mono_depth[2, 70, 100] *= 1e4
    assert bool(sc.mask[2, 70, 100])
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    align = ops.AlignOptions(min_correspondences=10**6, adaptive_correspondences=False, zero_unmasked_passthrough=True)
    res = DensifyEngine(DensifyConfig(voxel=0.1, align=align)).run(*_scene_args(sc, nbr))
    assert _status(res) == _lib.GRID_HASHED
    kx, krgb = _kept(res)
    _assert_oracle_voxels(*_voxels(res)[:4], kx, krgb, 0.1, list(res.host_grid().origin))


def test_steps_in_sequence_leave_the_table_clean(lib_built):
    """dense, hashed, hashed, dense on one engine: each step equals a fresh engine's."""
    from depthdensifier_b200 import _lib

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    args = _scene_args(sc, nbr)
    eng = _engine(max_cells=1 << 26, voxel=0.05, dedup_sparse=True)
    for voxel, status in [(0.05, _lib.GRID_OK), (0.02, _lib.GRID_HASHED), (0.015, _lib.GRID_HASHED), (0.05, _lib.GRID_OK)]:
        eng.cfg.voxel = voxel
        res = eng.run(*args)
        assert _status(res) == status
        fresh = _engine(max_cells=1 << 26, voxel=voxel, dedup_sparse=True).run(*args)
        for x, y in zip(_voxels(res), _voxels(fresh)):
            assert np.array_equal(x, y)
    assert bool((eng._hash.table == 255).all())  # every slot empty again


def test_axis_over_21_bits_still_raises(lib_built):
    from depthdensifier_b200 import _lib, ops

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    eng = _engine(voxel=1e-6)
    with pytest.raises(ops.DDNError, match="3x21-bit voxel key"):
        eng.run(*_scene_args(sc, nbr))
    assert eng.session().grid_state().status == _lib.GRID_TOO_MANY_BITS


def test_pipeline_main_on_a_dome_scene(lib_built, tmp_path):
    """pipeline.main with --fusion.voxel-size on a COLMAP model of an unbounded scene writes the oracle's voxels."""
    from depthdensifier_b200 import pipeline as P
    from depthdensifier_b200.colmap_io import Reconstruction
    from test_gpu_pipeline import _write_scene

    sc = make_scene(SceneConfig(**DOME))
    g = {k: getattr(sc, k).numpy() for k in ("mono_depth", "normal", "mask", "rgb", "cam_from_world", "intrinsics", "sparse_xyz",
                                              "sparse_offsets")}
    rec = _write_scene(tmp_path, g)
    cfg = P.ScriptConfig()
    cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images", output_model_dir=tmp_path / "out",
                              depth_dir=tmp_path / "depth")
    cfg.processing.downsample_density = 1
    cfg.refiner.adaptive_correspondences = False
    cfg.filtering.num_neighbours = 4
    cfg.filtering.neighbour_mode = "nearest"
    cfg.filtering.vote_threshold = default_vote_threshold(4)
    cfg.fusion.voxel_size = DOME_VOXEL
    out = P.main(cfg, return_candidates=True)
    # the device origin of the same step (the engine pipeline.main runs, on the same maps)
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    res = _engine(voxel=DOME_VOXEL).run(*_scene_args(sc, nbr))
    kept = out.candidates[out.keep].astype(np.float32)
    uk, mean, col, c = R.voxel_fuse(kept, np.zeros((len(kept), 3), np.uint8), DOME_VOXEL, np.array(list(res.host_grid().origin), np.float32))
    assert len(out.points) == len(uk) > 0
    assert np.abs(out.points - mean).max() <= 1e-5 * max(1.0, float(np.abs(mean).max()))
    back = Reconstruction()
    back.read_binary(tmp_path / "out")
    assert back.num_points3D() == rec.num_points3D() + len(uk)
