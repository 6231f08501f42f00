"""Oriented normals on the GPU: ddn_point_normals against the float64 statement of tests/normal_oracle.py, the fused
normals of every fusion path bit for bit against numpy from the kernels' own per-point normals, and the driver's PLY."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_mixed_scene, make_scene

import cpu_backend as CB
import normal_oracle as NO

pytestmark = pytest.mark.gpu

VOXEL = 0.02
K = 4
TOL = 2e-6


def _nbr(poses):
    return torch.from_numpy(nearest_views_table(poses, K).astype(np.int32)).cuda()


def _inputs(sc, depth=None):
    return ((sc.mono_depth if depth is None else depth).cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.cam_from_world.cuda(),
            sc.intrinsics.cuda(), sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), _nbr(sc.cam_from_world.numpy()))


def _run(sc, depth=None, **cfg):
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine
    from depthdensifier_b200.ops import FilterOptions

    stride = cfg.pop("stride", 1)
    eng = DensifyEngine(DensifyConfig(filter=FilterOptions(stride=stride), **cfg), device="cuda")
    res = eng.run(*_inputs(sc, depth))
    torch.cuda.synchronize()
    return res


@pytest.fixture(scope="module")
def scene():
    return make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))


def _assert_point_normals(got, ref, tie, votes):
    """Within TOL per component; an orientation tie may take either sign; no point: exactly 0."""
    got = got.astype(np.float64)
    err = np.abs(got - ref).max(-1)
    flip = np.abs(got + ref).max(-1)
    ok = (err <= TOL) | (tie & (flip <= TOL))
    assert ok.all(), f"{(~ok).sum()} normals differ, worst {err[~ok].max()}"
    assert (got[votes == 255] == 0).all()
    live = votes != 255
    assert live.any() and (np.abs(np.linalg.norm(got[live], axis=-1) - 1) <= 1e-5).all()


@pytest.mark.parametrize("stride", [1, 3])
def test_point_normals_uniform(lib_built, scene, stride):
    res = _run(scene, voxel=None, fuse_normals=True, stride=stride)
    votes = res.votes.cpu().numpy()
    ref, tie = NO.point_normals(scene.normal.numpy(), scene.cam_from_world.numpy(), scene.intrinsics.numpy(), votes, stride)
    got = res.normals.cpu().numpy()
    assert got.shape == votes.shape + (3,)
    for v in range(scene.n_views):
        _assert_point_normals(got[v], ref[v], tie[v], votes[v])


def test_point_normals_flip_sign_convention(lib_built, scene):
    """Normal maps with the opposite sign convention give the same oriented normals."""
    from depthdensifier_b200 import ops

    res = _run(scene, voxel=None, fuse_normals=True)
    flipped = ops.point_normals((-scene.normal).cuda().contiguous(), scene.cam_from_world.cuda(), scene.intrinsics.cuda(), res.votes, 1)
    votes = res.votes.cpu().numpy()
    _, tie = NO.point_normals(scene.normal.numpy(), scene.cam_from_world.numpy(), scene.intrinsics.numpy(), votes, 1)
    a, b = res.normals.cpu().numpy(), flipped.cpu().numpy()
    same = (a == b).all(-1)
    assert (same | tie).all() and same.mean() > 0.99


@pytest.mark.parametrize("stride", [1, 3])
def test_point_normals_ragged(lib_built, stride):
    """A mixed-size scene through run_views (device normals, and pinned host normals: the same bits)."""
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine
    from depthdensifier_b200.ops import FilterOptions

    sizes = [(96, 128), (80, 112), (128, 96), (104, 140), (96, 128), (72, 100)]
    ms = make_mixed_scene(SceneConfig(n_sparse=500, seed=4), sizes)
    poses, intr = ms.cam_from_world.numpy(), ms.intrinsics.numpy()
    eng = DensifyEngine(DensifyConfig(voxel=VOXEL, fuse_normals=True, filter=FilterOptions(stride=stride)), device="cuda")
    outs = []
    for normals in ([n.cuda() for n in ms.normal], list(ms.normal)):
        res = eng.run_views([d.cuda() for d in ms.mono_depth], normals, [m.cuda() for m in ms.mask], [c.cuda() for c in ms.rgb],
                            ms.cam_from_world.cuda(), ms.intrinsics.cuda(), ms.sparse_xyz.cuda(), ms.sparse_offsets.cuda(), _nbr(poses))
        torch.cuda.synchronize()
        outs.append(res)
    res = outs[0]
    assert torch.equal(res.normals, outs[1].normals) and torch.equal(res.voxel_normal, outs[1].voxel_normal)
    votes = [v.cpu().numpy() for v in res.per_view("votes")]
    ref, tie = NO.point_normals([n.numpy() for n in ms.normal], poses, intr, votes, stride)
    got = [n.cpu().numpy() for n in res.per_view("normals")]
    for v in range(len(sizes)):
        _assert_point_normals(got[v], ref[v], tie[v], votes[v])
    _assert_fused(res)


def _assert_fused(res, dedup=None):
    """The step's voxel keys and normals against numpy from its own kept points and per-point normals."""
    keep = res.keep_mask().reshape(-1).cpu().numpy()
    xyz = res.xyz.reshape(-1, 3).cpu().numpy()[keep]
    nrm = res.normals.reshape(-1, 3).cpu().numpy()[keep]
    g = res.host_grid()
    voxel, origin = np.float32(g.voxel), np.array(list(g.origin), np.float32)
    if dedup is not None:
        _, drop = CB.canonical_keys(dedup.astype(np.float32), voxel, origin)
        _, keys = CB.canonical_keys(xyz, voxel, origin)
        xyz, nrm = xyz[~np.isin(keys, drop)], nrm[~np.isin(keys, drop)]
    keys, sums = NO.fused_normal_sums(xyz, nrm, voxel, origin)
    assert len(keys) > 100
    assert np.array_equal(res.voxel_keys.cpu().numpy(), keys)
    got = res.voxel_normal.cpu().numpy()
    assert np.array_equal(got, NO.final_normals(sums))
    return keys, sums


@pytest.mark.parametrize("case", ["plain", "dedup", "support"])
def test_fused_normals_dense_and_hashed(lib_built, scene, case):
    """Dense session, hashed session (max_grid_cells = 2^16) and host-grid voxel_fuse on a grid within 2^35 cells and on one
    beyond it: the same keys and bit-identical normals, equal to the numpy statement."""
    from depthdensifier_b200 import ops

    kw = {"plain": {}, "dedup": {"dedup_sparse": True}, "support": {"min_support": 2, "support_tau": 0.01}}[case]
    dense = _run(scene, voxel=VOXEL, fuse_normals=True, **kw)
    hashed = _run(scene, voxel=VOXEL, fuse_normals=True, max_grid_cells=1 << 16, **kw)
    assert not dense.hash.ran() and hashed.hash.ran()
    dedup = scene.sparse_xyz.numpy() if case == "dedup" else None
    keys, _ = _assert_fused(dense, dedup)
    _assert_fused(hashed, dedup)
    assert torch.equal(dense.voxel_keys, hashed.voxel_keys) and torch.equal(dense.voxel_normal, hashed.voxel_normal)
    if case != "plain":
        return
    from depthdensifier_b200 import _lib

    g = dense.host_grid()
    big = _lib.VoxelGrid()
    big.voxel = g.voxel
    for i in range(3):
        big.origin[i], big.bits[i], big.dims[i] = g.origin[i], 12, 0  # 2^36 cells: the hashed kernels
    xyz, rgb, votes = dense.xyz.reshape(-1, 3), dense.grid_rgb().reshape(-1, 3), dense.votes.reshape(-1)
    normal = dense.normals.reshape(-1, 3)
    for grid in (g, big):
        k, x, c, n, nrm, counts = ops.voxel_fuse(xyz, rgb, votes, dense.fusion_threshold(), grid, row_len=dense.xyz.shape[2], normal=normal)
        assert torch.equal(k, dense.voxel_keys) and torch.equal(nrm, dense.voxel_normal)
        assert torch.equal(x, dense.voxel_xyz) and torch.equal(c, dense.voxel_rgb) and torch.equal(n, dense.voxel_count)
        k0, x0, c0, n0, counts0 = ops.voxel_fuse(xyz, rgb, votes, dense.fusion_threshold(), grid, row_len=dense.xyz.shape[2])
        assert torch.equal(k0, k) and torch.equal(x0, x) and torch.equal(counts0, counts)


@pytest.mark.parametrize("hashed", [False, True], ids=["dense", "hashed"])
def test_nothing_else_changes(lib_built, scene, hashed):
    kw = dict(voxel=VOXEL, min_support=1, dedup_sparse=True)
    if hashed:
        kw["max_grid_cells"] = 1 << 16
    off, on = _run(scene, **kw), _run(scene, fuse_normals=True, **kw)
    assert off.normals is None and off.voxel_normal is None
    for name in ("refined", "stats", "xyz", "votes", "support", "voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts", "bbox"):
        a, b = getattr(off, name), getattr(on, name)
        assert a.dtype == b.dtype and torch.equal(a, b), name


def test_ground_plane_accuracy(lib_built, scene):
    """With exact depths, voxels on the ground plane away from the spheres fuse to (0, 0, 1)."""
    res = _run(scene, depth=scene.true_depth, voxel=VOXEL, fuse_normals=True)
    x, n = res.voxel_xyz.cpu().numpy(), res.voxel_normal.cpu().numpy()
    far = np.ones(len(x), bool)
    for cx, cy, _, r in ((0.0, 0.0, 0.8, 0.8), (1.5, 0.5, 0.4, 0.4), (-1.2, -0.8, 0.5, 0.5)):
        far &= np.hypot(x[:, 0] - cx, x[:, 1] - cy) > r + 0.1
    plane = far & (np.abs(x[:, 2]) < VOXEL / 2)
    assert plane.sum() > 100
    assert np.abs(n[plane] - np.array([0, 0, 1], np.float32)).max() <= 1e-3
    assert (np.abs(np.linalg.norm(n, axis=1) - 1) <= 1e-6).all()


def test_driver_writes_oriented_ply(lib_built, golden_dir, tmp_path):
    from depthdensifier_b200 import pipeline as P
    from depthdensifier_b200.colmap_io import Reconstruction

    from test_gpu_pipeline import _write_scene
    from test_ply import read_ply

    g = np.load(golden_dir / "ref_main_allviews.npz")
    _write_scene(tmp_path, g)
    for voxel in (None, 0.05):
        cfg = P.ScriptConfig()
        ply = tmp_path / f"ply{voxel}" / "points3D.ply"
        cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images", output_model_dir=tmp_path / f"out{voxel}",
                                  depth_dir=tmp_path / "depth", output_ply=ply)
        cfg.processing.downsample_density = 2
        cfg.filtering.num_neighbours = 3
        cfg.fusion.voxel_size = voxel
        out = P.main(cfg)
        back = Reconstruction(tmp_path / f"out{voxel}")
        xyz, nrm, rgb = read_ply(ply)
        assert len(xyz) == back.num_points3D() == len(g["sparse_xyz"]) + len(out.points)
        ns = len(back.points3D)
        sp = [back.points3D[i] for i in sorted(back.points3D)]
        assert np.array_equal(xyz[:ns], np.array([p.xyz for p in sp], np.float32)) and (nrm[:ns] == 0).all()
        assert np.array_equal(rgb[:ns], np.array([p.color for p in sp], np.uint8))
        assert np.array_equal(xyz[ns:], out.points.astype(np.float32)) and np.array_equal(rgb[ns:], out.colors)
        assert np.array_equal(nrm[ns:], out.normals)
        lens = np.linalg.norm(nrm[ns:], axis=1)
        assert len(lens) > 0 and ((np.abs(lens - 1) <= 1e-5) | (lens == 0)).all() and (lens > 0).mean() > 0.99
