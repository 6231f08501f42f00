"""The main()-compatible driver and the reference's two helper functions, on the GPU, against the
reference's own outputs (tests/golden/ref_main_allviews.npz = unmodified scripts/test.py:main on these inputs)."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.colmap_io import Camera, Image, Reconstruction, Track, rotmat_to_quat
from oracle import restatement as R

pytestmark = pytest.mark.gpu


def _write_scene(tmp_path, g):
    """COLMAP model + images + precomputed depth maps from the golden arrays."""
    from PIL import Image as PILImage

    V, H, W = g["mono_depth"].shape
    rec = Reconstruction()
    off = g["sparse_offsets"]
    (tmp_path / "images").mkdir()
    (tmp_path / "depth").mkdir()
    for v in range(V):
        fx, fy, cx, cy = g["intrinsics"][v]
        rec.add_camera(Camera(v + 1, "PINHOLE", W, H, [fx, fy, cx, cy]))
        pose = g["cam_from_world"][v]
        ids = []
        for xyz in g["sparse_xyz"][off[v]:off[v + 1]]:
            ids.append(rec.add_point3D(xyz, Track([v + 1], [len(ids)]), (128, 128, 128)))
        n = len(ids)
        rec.add_image(Image(v + 1, rotmat_to_quat(pose[:, :3]), pose[:, 3], v + 1, f"view_{v:03d}.png", np.zeros((n, 2)), ids))
        PILImage.fromarray(g["rgb"][v]).save(tmp_path / "images" / f"view_{v:03d}.png")
        np.savez(tmp_path / "depth" / f"view_{v:03d}.npz", depth=g["mono_depth"][v], normal=g["normal"][v], mask=g["mask"][v])
    rec.write_binary(tmp_path / "sparse")
    return rec


def test_main_matches_reference_main(lib_built, golden_dir, tmp_path):
    from depthdensifier_b200 import pipeline as P

    g = np.load(golden_dir / "ref_main_allviews.npz")
    _write_scene(tmp_path, g)
    cfg = P.ScriptConfig()
    cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images", output_model_dir=tmp_path / "out",
                              depth_dir=tmp_path / "depth")
    cfg.processing.downsample_density = 1
    cfg.refiner.adaptive_correspondences = False  # the golden run has no random subsample
    cfg.filtering.vote_threshold = int(g["vote_threshold"])
    out = P.main(cfg, return_candidates=True)
    ref_pts, ref_keep = g["ref_points"], g["ref_keep"]
    assert out.num_candidates == len(ref_pts)
    scale = max(1.0, np.abs(ref_pts).max())
    assert np.abs(out.candidates - ref_pts).max() <= 1e-5 * scale
    assert (out.keep != ref_keep).mean() < 0.005  # threshold ties only (exact tie-band comparison: test_gpu_parity)
    both = out.keep & ref_keep
    sel_mine = both[out.keep]
    sel_ref = both[ref_keep]
    # the reference's kept cloud is its candidates at `keep` (make_golden.py checks that when it records the file)
    assert np.abs(out.points[sel_mine] - ref_pts[ref_keep][sel_ref]).max() <= 1e-5 * scale
    assert np.array_equal(out.colors[sel_mine], g["ref_colors"][ref_keep][sel_ref])
    # the written model: sparse points retained, dense points appended (scripts/test.py:353-364)
    back = Reconstruction(tmp_path / "out")
    assert len(back.points3D) == len(g["sparse_xyz"]) and back.num_dense_points() == len(out.points)
    dx, dc = back.dense_points()
    assert np.array_equal(dx, out.points) and np.array_equal(dc, out.colors)
    assert back.num_reg_images() == g["mono_depth"].shape[0]


def test_main_north_star_settings(lib_built, golden_dir, tmp_path):
    """K nearest neighbours + voxel fusion through the same entry point."""
    from depthdensifier_b200 import pipeline as P

    g = np.load(golden_dir / "ref_main_allviews.npz")
    _write_scene(tmp_path, g)
    cfg = P.ScriptConfig()
    cfg.paths = P.PathsConfig(recon_path=tmp_path / "sparse", image_dir=tmp_path / "images", output_model_dir=tmp_path / "out",
                              depth_dir=tmp_path / "depth")
    cfg.processing.downsample_density = 2
    cfg.filtering.num_neighbours = 3
    cfg.filtering.vote_threshold = 2
    cfg.fusion.voxel_size = 0.05
    out = P.main(cfg, return_candidates=True)
    kept = out.candidates[out.keep].astype(np.float32)
    keys_ref = np.unique(R.voxel_keys(kept, 0.05, R.voxel_origin(kept, 0.05)))
    assert len(out.points) == len(keys_ref) and 0 < len(out.points) < out.keep.sum()


def test_project_unproject_helpers(lib_built):
    from depthdensifier_b200 import pipeline as P

    rng = np.random.default_rng(0)
    q = rng.normal(size=4)
    from depthdensifier_b200.colmap_io import quat_to_rotmat

    Rm, t = quat_to_rotmat(q), rng.normal(size=3)
    image = Image(1, rotmat_to_quat(Rm), t, 1, "x.png")
    cam = Camera(1, "PINHOLE", 640, 480, [510.5, 498.25, 321.0, 239.5])
    pts = rng.normal(size=(1000, 3)) * 3
    uv, z = P.project_points(pts, image, cam)
    uv_ref, z_ref = R.project_points(pts, image.cam_from_world().matrix(), cam.calibration_matrix())
    assert np.allclose(z, z_ref, rtol=1e-13, atol=1e-13) and np.allclose(uv, uv_ref, rtol=1e-11, atol=1e-9)
    px = np.stack([rng.integers(0, 640, 500), rng.integers(0, 480, 500)], -1)
    d = rng.uniform(0.5, 9, 500).astype(np.float32)
    got = P.unproject_points(px, d, cam)
    fx, fy, cx, cy = cam.params
    ref = np.stack([(px[:, 0] - cx) / fx * d, (px[:, 1] - cy) / fy * d, d], -1)  # scripts/test.py:81-89
    assert got.dtype == np.float64 and np.array_equal(got, ref)
    assert P.unproject_points(np.zeros((0, 2)), np.zeros(0, np.float32), cam).shape == (0, 3)
