"""Edge cases of the hot path on the GPU: empty and degenerate inputs, padded / duplicated neighbour tables,
randomised voxel fusion (hypothesis) against the numpy definition."""

import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings
from hypothesis import strategies as st

from depthdensifier_b200.neighbours import nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import parity

pytestmark = pytest.mark.gpu


def _cuda(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def test_fuse_empty_and_fully_rejected(lib_built):
    """Empty input, all points rejected, points outside the grid, empty partials and an empty merge."""
    _check_empty_and_rejected(large=False)


def test_fuse_empty_and_fully_rejected_over_2e35_cells(lib_built):
    """The same on a grid of more than 2^35 cells (hashed path)."""
    _check_empty_and_rejected(large=True)


def _check_empty_and_rejected(large: bool):
    from depthdensifier_b200 import ops

    grid = ops.make_grid([0, 0, 0], [100, 100, 100], 0.01) if large else ops.make_grid([0, 0, 0], [1, 1, 1], 0.1)
    assert (ops.fuse_tile_info(grid)[0] == 0) == large
    e = ops.voxel_fuse(torch.zeros((0, 3), device="cuda"), torch.zeros((0, 3), dtype=torch.uint8, device="cuda"), None, 1, grid)
    assert e[4].cpu().tolist() == [0, 0] and all(len(t) == 0 for t in e[:4])
    xyz = _cuda(np.random.default_rng(0).uniform(0, 1, (1000, 3)).astype(np.float32))
    rgb = _cuda(np.zeros((1000, 3), np.uint8))
    votes = torch.full((1000,), 255, dtype=torch.uint8, device="cuda")  # nothing participates
    k, x, c, n, counts = ops.voxel_fuse(xyz, rgb, votes, 3, grid)
    assert counts.cpu().tolist() == [0, 0] and len(k) == 0
    # points outside the grid do not participate either
    far = xyz + 1000.0
    k, x, c, n, counts = ops.voxel_fuse(far, rgb, None, 1, grid)
    assert counts.cpu().tolist() == [0, 0]
    rec, cnt = ops.voxel_fuse_partial(xyz, rgb, votes, 3, grid)
    assert cnt.cpu().tolist() == [0, 0]
    m = ops.voxel_merge_partials(torch.zeros((0, 6), dtype=torch.int64, device="cuda"), grid, trim=True)
    assert m[4].cpu().tolist() == [0, 0]


@settings(max_examples=25, deadline=None, derandomize=True, suppress_health_check=[HealthCheck.function_scoped_fixture])
@given(n=st.integers(1, 3000), voxel=st.sampled_from([0.5, 0.1, 0.03]), seed=st.integers(0, 10_000),
       row_len=st.sampled_from([0, 8, 13, 64]), clustered=st.booleans(), far=st.booleans())
def test_fuse_random_vs_numpy(lib_built, n, voxel, seed, row_len, clustered, far):
    """far: a quarter of the points (at least one) 4 km away, so the grid has more than 2^35 cells (hashed path)."""
    from depthdensifier_b200 import ops

    rng = np.random.default_rng(seed)
    xyz = (rng.normal(0, 0.02 if clustered else 1.0, (n, 3)) + rng.uniform(-3, 3, 3)).astype(np.float32)
    if far:
        xyz[: max(1, n // 4)] += np.float32(4000.0)
    rgb = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    origin = R.voxel_origin(xyz, voxel)
    k_ref, m_ref, c_ref, n_ref = R.voxel_fuse(xyz, rgb, voxel, origin)
    grid = ops.make_grid(xyz.min(0), xyz.max(0), voxel)
    k, m, c, cnt, counts = ops.voxel_fuse(_cuda(xyz), _cuda(rgb), None, 1, grid, row_len=row_len)
    assert counts.cpu().tolist() == [n, len(k_ref)]
    assert np.array_equal(k.cpu().numpy().view(np.uint64), k_ref) and np.array_equal(cnt.cpu().numpy(), n_ref)
    assert np.array_equal(c.cpu().numpy(), c_ref)
    assert np.abs(m.cpu().numpy() - m_ref).max() <= 1e-5 * max(1.0, np.abs(m_ref).max())


@pytest.mark.parametrize("large", [False, True], ids=["dense", "over_2e35_cells"])
def test_fuse_flags_a_voxel_of_2e24_points(lib_built, large):
    """A voxel that collects 2^24 points (32-bit colour sums) sets counts[0] = -1 on every grid, and trim raises."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200._lib import DDNError

    grid = ops.make_grid([0, 0, 0], [100, 100, 100], 0.01) if large else ops.make_grid([0, 0, 0], [1, 1, 1], 0.1)
    assert (ops.fuse_tile_info(grid)[0] == 0) == large
    n = 1 << 24
    xyz = torch.full((n, 3), 0.555, dtype=torch.float32, device="cuda")
    rgb = torch.full((n, 3), 255, dtype=torch.uint8, device="cuda")
    counts = ops.voxel_fuse(xyz, rgb, None, 1, grid, trim=False)[4]
    assert counts.cpu().tolist() == [-1, 1]
    with pytest.raises(DDNError, match="2\\^24"):
        ops.voxel_fuse(xyz, rgb, None, 1, grid, trim=True)


def test_filter_padded_and_duplicate_neighbours(lib_built):
    """-1 entries are skipped, a neighbour listed twice votes twice, the own view may appear anywhere."""
    from depthdensifier_b200 import ops

    sc = make_scene(SceneConfig(n_views=5, width=120, height=90, n_sparse=600, seed=11))
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    refined = sc.mono_depth.numpy() * sc.mask.numpy()  # any depth maps will do for stage 3
    nbr = np.array([[1, -1, 2, 2, 0, -1], [-1, -1, -1, -1, -1, -1], [3, 3, 3, 1, -1, 4], [0, 1, 2, 3, 4, -1], [4, 4, 0, -1, 1, 2]],
                   np.int32)
    d_pose, d_intr, d_nbr = _cuda(poses), _cuda(intr), _cuda(nbr)
    pair, src = ops.build_pair_tables(d_pose, d_intr, d_nbr, 0, 5, 90, 120)
    xyz, votes = ops.backproject_filter(_cuda(refined), _cuda(sc.normal.numpy()), d_nbr, pair, src, 0, 2, ops.FilterOptions())
    votes = votes.cpu().numpy()
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    assert (votes[1][valid[1]] == 0).all()  # a view without neighbours collects no votes
    vv = np.nonzero(valid)[0]
    pts = np.concatenate([R.backproject_view(refined[v], intr[v], poses[v])[0] for v in range(5)])
    nrm = sc.normal.numpy()[valid]
    ref_votes = np.zeros(len(pts), np.int64)
    nties = np.zeros(len(pts), np.int64)
    for s in range(5):
        sel = np.where(vv == s)[0]
        for t in nbr[s]:
            if t >= 0:
                v_t, tie_t = parity.pair_ties(pts[sel], nrm[sel], vv[sel], int(t), refined[t], poses[t], intr[t])
                ref_votes[sel] += v_t
                nties[sel] += tie_t
    parity.assert_votes_match(votes[valid], ref_votes, nties, max_tie_fraction=0.05)
    assert ref_votes.max() >= 2  # the duplicated neighbours really vote twice somewhere


def test_align_degenerate_views(lib_built):
    """All-masked view, view with one sparse point, view whose sparse points are all behind the camera."""
    from depthdensifier_b200 import ops

    sc = make_scene(SceneConfig(n_views=4, width=96, height=64, n_sparse=300, seed=5))
    depth = sc.mono_depth.numpy().copy()
    mask = sc.mask.numpy().copy()
    mask[0] = False  # view 0: nothing to remap -> all zeros
    off = sc.sparse_offsets.numpy()
    sparse = sc.sparse_xyz.numpy().copy()
    poses = sc.cam_from_world.numpy()
    # view 2: move its sparse points behind the camera (z_cam < 0)
    Rm, t = poses[2][:, :3], poses[2][:, 3]
    cam = sparse[off[2]:off[3]] @ Rm.T + t
    cam[:, 2] = -np.abs(cam[:, 2]) - 1
    sparse[off[2]:off[3]] = (cam - t) @ Rm
    # view 3: a single sparse point
    keep = np.ones(len(sparse), bool)
    keep[off[3] + 1:off[4]] = False
    sparse2 = sparse[keep]
    off2 = off.copy()
    off2[4] = off[3] + 1
    kmat = np.stack([R.kmatrix(i) for i in sc.intrinsics.numpy()])
    refined, stats = ops.align_views(_cuda(depth), _cuda(mask), _cuda(poses), _cuda(kmat), _cuda(sparse2), _cuda(off2), 300,
                                     ops.AlignOptions(zero_unmasked_passthrough=True))
    st_ = ops.decode_stats(stats)
    refined = refined.cpu().numpy()
    assert (refined[0] == 0).all()
    assert st_[1]["status"] == 0
    assert st_[2]["status"] == 1 and np.array_equal(refined[2], np.where(mask[2], depth[2], 0))  # passthrough, masked
    assert st_[3]["status"] in (1, 2, 3) and np.array_equal(refined[3], np.where(mask[3], depth[3], 0))
    for v in (2, 3):  # the oracle agrees these views are returned unchanged
        lo, hi = int(off2[v]), int(off2[v + 1])
        r = R.refine_view(depth[v].copy(), sparse2[lo:hi], poses[v], kmat[v], mask[v])
        assert "outliers_removed" not in r
