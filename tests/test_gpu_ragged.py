"""Views of different sizes on the GPU (the ragged layout, include/ddn_b200.h DDN_LAYOUT_COLS).

Uniform scenes through the ragged path must give the uniform path's bits.  Mixed sizes have no golden vectors from the
reference (no mixed-size run of it is recorded): their parity rests on the oracle's per-view list form
(tests/ragged_oracle.py, built from oracle/restatement.py's per-view functions), which follows the reference's per-image
loop and takes every view at its own size, compared with the bars the other parity tests use."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import all_views_table, default_vote_threshold, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_mixed_scene, make_scene
from oracle import restatement as R

import parity
import ragged_oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _engine(voxel=0.02, dedup=False, thr=None, **fopts):
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    align = ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True)
    return DensifyEngine(DensifyConfig(align=align, filter=ops.FilterOptions(**fopts), vote_threshold=thr, voxel=voxel,
                                       dedup_sparse=dedup))


@pytest.mark.parametrize("sample_mode,tau,stride,table,pixel_layout", [
    ("nearest", 0.0, 1, "all", 0),
    ("nearest", 0.0, 3, "knn", 1),
    ("nearest", 0.05, 1, "knn", 0),
    ("bilinear", 0.0, 1, "knn", 1),
    ("bilinear", 0.05, 3, "all", 0),
])
def test_uniform_scene_through_ragged_path_is_bit_identical(lib_built, sample_mode, tau, stride, table, pixel_layout):
    sc = make_scene(SceneConfig(n_views=6, width=131, height=77, n_sparse=400, seed=3), "cuda")
    V = sc.n_views
    nbr = all_views_table(V) if table == "all" else nearest_views_table(sc.cam_from_world.cpu().numpy(), 3)
    nbr = torch.from_numpy(nbr.astype(np.int32)).cuda()
    eng = _engine(sample_mode=sample_mode, two_sided_tau=tau, stride=stride, pixel_layout=pixel_layout)
    args = (sc.cam_from_world, sc.intrinsics, sc.sparse_xyz, sc.sparse_offsets, nbr)
    a = eng.run(sc.mono_depth, sc.normal, sc.mask, sc.rgb, *args)
    b = eng.run_views(list(sc.mono_depth), list(sc.normal), list(sc.mask), list(sc.rgb), *args)
    assert a.check() > 0 and b.layout.stride == stride
    assert torch.equal(a.refined.view(-1), b.refined) and torch.equal(a.stats, b.stats)
    assert torch.equal(a.xyz.view(-1, 3), b.xyz) and torch.equal(a.votes.view(-1), b.votes)
    assert int((a.votes != 255).sum()) > 0 and int(a.votes[a.votes != 255].max()) >= 1
    assert torch.equal(a.bbox, b.bbox) and torch.equal(a.bbox_valid, b.bbox_valid)
    assert torch.equal(a.keep_mask().view(-1), b.keep_mask())
    assert list(a.host_grid().origin) == list(b.host_grid().origin)
    for f in ("voxel_keys", "voxel_xyz", "voxel_rgb", "voxel_count", "counts"):
        assert torch.equal(getattr(a, f), getattr(b, f)), f
    assert all(torch.equal(x, y) for x, y in zip(a.per_view("xyz"), b.per_view("xyz")))


# portrait and landscape, odd sides, a view smaller than one consistency chunk (20 x 30 = 600 points), a 2-row view
MIXED_SIZES = [(77, 131), (131, 77), (64, 96), (96, 64), (2, 150), (20, 30), (101, 127), (45, 63)]
NO_SPARSE_VIEW = 3


def _mixed(seed=17):
    ms = make_mixed_scene(SceneConfig(n_sparse=400, seed=seed), MIXED_SIZES)
    off = ms.sparse_offsets.numpy().copy()
    lo, hi = off[NO_SPARSE_VIEW], off[NO_SPARSE_VIEW + 1]  # one view without sparse points (scripts/test.py:136-137)
    keep = np.ones(len(ms.sparse_xyz), bool)
    keep[lo:hi] = False
    off[NO_SPARSE_VIEW + 1:] -= hi - lo
    return ms, ms.sparse_xyz.numpy()[keep], off


def _votes_with_ties(points, normals, src_view, refined, poses, intr, nbr, active, sample_mode, **kw):
    """parity.votes_with_ties for per-view maps of their own sizes (pair_ties* take one target map each)."""
    V = len(refined)
    votes = np.zeros(len(points), np.int64)
    nties = np.zeros(len(points), np.int64)
    member = np.zeros((V, V), bool)
    for s in range(V):
        member[s, nbr[s][nbr[s] >= 0]] = True
    fn = parity.pair_ties if sample_mode == "nearest" else parity.pair_ties_bilinear
    for t in active:
        sel = np.where(member[src_view, t])[0]
        if len(sel):
            vt, tt = fn(points[sel], normals[sel], src_view[sel], t, refined[t], poses[t], intr[t], **kw)
            votes[sel] += vt
            nties[sel] += tt
    return votes, nties


@pytest.mark.parametrize("K,dedup,sample_mode,stride", [(None, False, "nearest", 1), (3, True, "nearest", 2), (3, False, "bilinear", 1)],
                         ids=["K=V", "K<V-dedup-stride2", "K<V-bilinear"])
def test_mixed_sizes_match_the_oracle(lib_built, K, dedup, sample_mode, stride):
    ms, sparse, off = _mixed()
    V = ms.n_views
    poses, intr = ms.cam_from_world.numpy(), ms.intrinsics.numpy()
    nbr = all_views_table(V) if K is None else nearest_views_table(poses, K)
    thr = 3 if K is None else default_vote_threshold(K)
    voxel = 0.03
    maps = [[m.numpy() for m in x] for x in (ms.mono_depth, ms.normal, ms.mask, ms.rgb)]
    out = ragged_oracle.densify_views(*maps, sparse, off, poses, intr, nbr, thr, align=R.AlignConfig(adaptive_correspondences=False), stride=stride,
                    sample_mode=sample_mode)
    cuda = lambda x: torch.as_tensor(np.ascontiguousarray(x)).cuda()
    eng = _engine(voxel=voxel, dedup=dedup, thr=thr, sample_mode=sample_mode, stride=stride)
    res = eng.run_views([cuda(m) for m in maps[0]], [cuda(m) for m in maps[1]], [cuda(m) for m in maps[2]], [cuda(m) for m in maps[3]],
                        cuda(poses), cuda(intr), cuda(sparse), cuda(off), cuda(nbr.astype(np.int32)))
    res.check()
    from depthdensifier_b200 import ops

    st = ops.decode_stats(res.stats)
    assert st[NO_SPARSE_VIEW]["status"] == 5 and sum(s["status"] == 0 for s in st) >= 4
    refined = [r.cpu().numpy() for r in res.per_view("refined")]
    for v in range(V):
        assert refined[v].shape == MIXED_SIZES[v]
        assert np.array_equal(refined[v] > 0, out["refined"][v] > 0), v
        np.testing.assert_allclose(refined[v], out["refined"][v], rtol=RTOL, atol=0, err_msg=f"view {v}")
    # back-projected points in the oracle's order (view by view, row-major on each strided grid)
    votes = res.votes.cpu().numpy()
    valid = votes != 255
    assert valid.sum() == len(out["points"])
    xyz = res.xyz.cpu().numpy()[valid]
    scale = max(1.0, np.abs(out["points"]).max())
    assert np.abs(xyz - out["points"]).max() <= RTOL * scale
    active = [int(v) for v in out["active_views"]]
    ref_votes, nties = _votes_with_ties(out["points"], out["normals"], out["src_view"], out["refined"], poses, intr, nbr, active,
                                        sample_mode)
    assert np.array_equal(ref_votes, out["votes"])  # the tie analysis reproduces the statement's own votes
    parity.assert_votes_match(votes[valid], ref_votes, nties, max_tie_fraction=0.02 if sample_mode == "nearest" else 0.08)
    assert out["votes"].max() >= 1
    keep_gpu = votes[valid] < thr
    clean = nties == 0
    assert np.array_equal(keep_gpu[clean], out["keep"][clean])
    # voxel fusion of the kept points, bit-exact against the oracle on the device grid
    origin = np.array(list(res.host_grid().origin), np.float32)
    k, m, c, n = R.voxel_fuse(xyz[keep_gpu].astype(np.float32), out["colors"][keep_gpu], voxel, origin)
    if dedup:
        s32 = sparse.astype(np.float32)
        k3 = np.floor((s32 - origin) / np.float32(voxel)).astype(np.int64)
        sk = (k3[:, 0] | (k3[:, 1] << 21) | (k3[:, 2] << 42)).astype(np.uint64)[((k3 >= 0) & (k3 < (1 << 21))).all(1)]
        drop = np.isin(k, sk)
        assert drop.any()
        k, m, c, n = k[~drop], m[~drop], c[~drop], n[~drop]
    assert np.array_equal(res.voxel_keys.cpu().numpy().view(np.uint64), k)
    assert np.array_equal(res.voxel_count.cpu().numpy(), n) and np.array_equal(res.voxel_rgb.cpu().numpy(), c)
    assert np.abs(res.voxel_xyz.cpu().numpy() - m).max() <= RTOL * scale


def _write_mixed_model(tmp_path, ms, sparse, off):
    """COLMAP model with two PINHOLE cameras (landscape views use camera 1, portrait views camera 2) + images + depth maps."""
    from PIL import Image as PILImage

    from depthdensifier_b200.colmap_io import Camera, Image, Reconstruction, Track, rotmat_to_quat

    rec = Reconstruction()
    (tmp_path / "images").mkdir()
    (tmp_path / "depth").mkdir()
    cams = {}
    for v, (h, w) in enumerate(ms.sizes):
        if (h, w) not in cams:
            cams[(h, w)] = len(cams) + 1
            rec.add_camera(Camera(cams[(h, w)], "PINHOLE", w, h, list(ms.intrinsics[v].numpy())))
        pose = ms.cam_from_world[v].numpy()
        ids = [rec.add_point3D(xyz, Track([v + 1], [i]), (128, 128, 128)) for i, xyz in enumerate(sparse[off[v]:off[v + 1]])]
        rec.add_image(Image(v + 1, rotmat_to_quat(pose[:, :3]), pose[:, 3], cams[(h, w)], f"view_{v:03d}.png", np.zeros((len(ids), 2)), ids))
        PILImage.fromarray(ms.rgb[v].numpy()).save(tmp_path / "images" / f"view_{v:03d}.png")
        np.savez(tmp_path / "depth" / f"view_{v:03d}.npz", depth=ms.mono_depth[v].numpy(), normal=ms.normal[v].numpy(),
                 mask=ms.mask[v].numpy())
    rec.write_binary(tmp_path / "sparse")
    assert len(cams) == 2


@pytest.mark.parametrize("factor", [1, 2])
def test_pipeline_main_two_cameras_of_different_sizes(lib_built, tmp_path, factor):
    from depthdensifier_b200 import pipeline as P
    from depthdensifier_b200.colmap_io import Reconstruction

    sizes = [(96, 128), (128, 96)] * 3
    ms = make_mixed_scene(SceneConfig(n_sparse=300, seed=23), sizes)
    sparse, off = ms.sparse_xyz.numpy(), ms.sparse_offsets.numpy()
    _write_mixed_model(tmp_path, ms, sparse, off)
    cfg = P.ScriptConfig()
    cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images", output_model_dir=tmp_path / "out",
                              depth_dir=tmp_path / "depth")
    cfg.processing.downsample_density = 2
    cfg.processing.pipeline_downsample_factor = factor
    cfg.refiner.adaptive_correspondences = False
    cfg.filtering.vote_threshold = 3
    if factor == 2:  # the provider sees the image at processing size: hand it the maps at that size
        (tmp_path / "depth2").mkdir()
        for v, (h, w) in enumerate(sizes):
            z = np.load(tmp_path / "depth" / f"view_{v:03d}.npz")
            np.savez(tmp_path / "depth2" / f"view_{v:03d}.npz", depth=z["depth"][::2, ::2], normal=z["normal"][::2, ::2],
                     mask=z["mask"][::2, ::2])
        cfg.paths.depth_dir = tmp_path / "depth2"
    out = P.main(cfg, return_candidates=True)
    # the same per-view arrays through the oracle
    rec = Reconstruction(tmp_path / "sparse")
    depths, normals, masks, rgbs, poses, intr = [], [], [], [], [], []
    from depthdensifier_b200.pipeline import load_image_rgb

    for v in range(len(sizes)):
        z = np.load(cfg.paths.depth_dir / f"view_{v:03d}.npz")
        depths.append(z["depth"].astype(np.float32)), normals.append(z["normal"].astype(np.float32)), masks.append(z["mask"])
        rgbs.append(load_image_rgb(tmp_path / "images" / f"view_{v:03d}.png", factor))
        im = rec.images[v + 1]
        cam = rec.cameras[im.camera_id]
        cam.rescale(new_width=rgbs[-1].shape[1], new_height=rgbs[-1].shape[0])
        poses.append(im.cam_from_world().matrix())
        intr.append(np.array(cam.params[:4], np.float64))
    poses, intr = np.stack(poses), np.stack(intr)
    ref = ragged_oracle.densify_views(depths, normals, masks, rgbs, sparse, off, poses, intr, all_views_table(len(sizes)), 3,
                    align=R.AlignConfig(adaptive_correspondences=False), stride=2)
    assert out.num_candidates == len(ref["points"]) > 0
    scale = max(1.0, np.abs(ref["points"]).max())
    assert np.abs(out.candidates - ref["points"]).max() <= RTOL * scale
    assert (out.keep != ref["keep"]).mean() < 0.005  # threshold ties only
    both = out.keep & ref["keep"]
    assert np.abs(out.points[both[out.keep]] - ref["points"][ref["keep"]][both[ref["keep"]]]).max() <= RTOL * scale
    assert np.array_equal(out.colors[both[out.keep]], ref["colors"][ref["keep"]][both[ref["keep"]]])
    assert ref["votes"].max() >= 1
    back = Reconstruction(tmp_path / "out")
    assert len(back.points3D) == len(sparse) and back.num_dense_points() == len(out.points)  # sparse retained, dense appended
    dx, dc = back.dense_points()
    assert np.array_equal(dx, out.points) and np.array_equal(dc, out.colors)
    assert back.num_reg_images() == len(sizes) and len(back.cameras) == 2
