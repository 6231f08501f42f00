"""The host statement of the oriented and fused normals (tests/normal_oracle.py) on hand-made cases, without a GPU."""

import numpy as np

import normal_oracle as NO

VOXEL = np.float32(0.1)
ORIGIN = np.zeros(3, np.float32)
EYE = np.concatenate([np.eye(3), np.zeros((3, 1))], 1)
INTR = (10.0, 10.0, 2.0, 2.0)  # fx, fy, cx, cy of a 5 x 5 view


def _view(n_c, pose=EYE, votes=None):
    nmap = np.broadcast_to(np.asarray(n_c, np.float32), (5, 5, 3)).copy()
    votes = np.zeros((5, 5), np.uint8) if votes is None else votes
    return NO.view_normals(nmap, pose, INTR, votes, 1)


def test_plane_fuses_to_its_normal():
    """A tilted plane seen by a rotated camera: every point's normal is the plane's, and so is the fused one."""
    a = 0.3
    Rz = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])  # cam_from_world rotation
    pose = np.concatenate([Rz, np.zeros((3, 1))], 1)
    world_n = np.array([0.0, 0.6, -0.8])
    n, tie = _view(Rz @ world_n, pose)
    assert not tie.any()
    np.testing.assert_allclose(n.reshape(-1, 3), np.tile(world_n, (25, 1)), atol=1e-7)
    rng = np.random.default_rng(0)
    xyz = (rng.uniform(0, 0.1, (25, 3))).astype(np.float32)  # one voxel
    keys, sums = NO.fused_normal_sums(xyz, n.reshape(-1, 3).astype(np.float32), VOXEL, ORIGIN)
    assert len(keys) == 1
    np.testing.assert_allclose(NO.final_normals(sums)[0], world_n, atol=1e-6)


def test_back_facing_normal_flips():
    """A normal along the viewing ray (n_c . r > 0) is negated; the opposite one is kept."""
    away, _ = _view((0.0, 0.0, 1.0))
    toward, _ = _view((0.0, 0.0, -1.0))
    np.testing.assert_allclose(away[2, 2], (0, 0, -1), atol=1e-8)
    np.testing.assert_allclose(toward[2, 2], (0, 0, -1), atol=1e-8)
    # off-centre pixel: the ray is (x - cx) / fx, ..., so a normal facing +x flips only right of the centre
    side, tie = _view((1.0, 0.0, 0.0))
    assert side[2, 4, 0] < 0 and side[2, 0, 0] > 0 and tie[2, 2] and not tie[2, 4]


def test_zero_nan_and_missing_points():
    """Zero and NaN normals, and grid points without a point, are (0, 0, 0): they add nothing to a voxel's sum but the
    points still count in it."""
    nmap = np.zeros((5, 5, 3), np.float32)
    nmap[..., 2] = -1
    nmap[0, 0] = 0
    nmap[0, 1] = (np.nan, 0, -1)
    nmap[0, 2] = (0, np.inf, -1)
    votes = np.zeros((5, 5), np.uint8)
    votes[0, 3] = 255
    n, _ = NO.view_normals(nmap, EYE, INTR, votes, 1)
    for x in range(4):
        assert np.array_equal(n[0, x], np.zeros(3)), x
    np.testing.assert_allclose(n[0, 4], (0, 0, -1), atol=1e-8)
    xyz = np.full((5, 3), 0.05, np.float32)
    keys, sums = NO.fused_normal_sums(xyz, n[0].astype(np.float32), VOXEL, ORIGIN)
    assert len(keys) == 1 and sums.tolist() == [[0, 0, -(1 << 20)]]
    np.testing.assert_array_equal(NO.final_normals(sums), [[0, 0, -1]])
    assert NO.final_normals(np.zeros((1, 3), np.int64)).tolist() == [[0, 0, 0]]


def test_strided_grid_uses_the_strided_pixel():
    nmap = np.zeros((7, 7, 3), np.float32)
    nmap[..., 2] = -1
    nmap[3, 6] = (0.6, 0, -0.8)  # grid point (x=2, y=1) at stride 3
    n, _ = NO.view_normals(nmap, EYE, INTR, np.zeros((3, 3), np.uint8), 3)
    np.testing.assert_allclose(n[1, 2], (0.6, 0, -0.8), atol=1e-7)


def test_sums_do_not_depend_on_point_order():
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0, 0.5, (2000, 3)).astype(np.float32)
    nrm = rng.normal(size=(2000, 3))
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    k0, s0 = NO.fused_normal_sums(xyz, nrm, VOXEL, ORIGIN)
    perm = rng.permutation(2000)
    k1, s1 = NO.fused_normal_sums(xyz[perm], nrm[perm], VOXEL, ORIGIN)
    assert np.array_equal(k0, k1) and np.array_equal(s0, s1)
    assert np.array_equal(NO.final_normals(s0), NO.final_normals(s1))
    q = NO.quantize(nrm)
    assert np.abs(q).max() <= 1 << 20 and NO.quantize(np.float32([[2.5 / (1 << 20), -0.5 / (1 << 20), 0]])).tolist() == [[2, 0, 0]]
