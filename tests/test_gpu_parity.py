"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden vectors
produced by the reference's own code.  Run with `pytest -m gpu` on a B200."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.hashperm import hash_perm
from depthdensifier_b200.neighbours import all_views_table, default_vote_threshold, nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import parity

pytestmark = pytest.mark.gpu

# float tolerances (stated): refined depth and positions within 1e-5 relative (north_star)
RTOL = 1e-5


def _cuda(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def _run_filter(refined_all, normal, poses, intr, nbr, thr, **fopts):
    from depthdensifier_b200 import ops

    V = refined_all.shape[0]
    d_ref = _cuda(refined_all)
    d_nrm = _cuda(normal)
    d_pose = _cuda(poses)
    d_intr = _cuda(intr)
    d_nbr = _cuda(nbr.astype(np.int32))
    pair, src = ops.build_pair_tables(d_pose, d_intr, d_nbr, 0, V, refined_all.shape[1], refined_all.shape[2])
    bbox = ops.new_bbox(d_ref.device)
    xyz, votes = ops.backproject_filter(d_ref, d_nrm, d_nbr, pair, src, 0, thr, ops.FilterOptions(**fopts), bbox=bbox)
    torch.cuda.synchronize()
    return xyz.cpu().numpy(), votes.cpu().numpy(), ops.decode_bbox(bbox)


def _assert_xyz_close(gpu, ref):
    scale = np.maximum(np.abs(ref).max(), 1.0)
    err = np.abs(gpu.astype(np.float64) - ref).max()
    assert err <= RTOL * scale, f"max abs position error {err} vs scale {scale}"


def test_filter_matches_reference_main_golden(lib_built, golden_dir):
    """K = V, own view included: the reference's exact semantics (scripts/test.py:273-330)."""
    g = np.load(golden_dir / "ref_main_allviews.npz")
    refined = g["ref_refined"]
    V = refined.shape[0]
    thr = int(g["vote_threshold"])
    xyz, votes, bbox = _run_filter(refined, g["normal"], g["cam_from_world"], g["intrinsics"], all_views_table(V), thr)
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    assert valid.sum() == len(g["ref_points"])
    _assert_xyz_close(xyz[valid], g["ref_points"])
    src = np.repeat(np.arange(V), valid.reshape(V, -1).sum(1)).astype(np.int32)
    ref_votes, nties = parity.votes_with_ties(g["ref_points"], g["ref_normals"], src, refined, g["cam_from_world"], g["intrinsics"], all_views_table(V))
    assert np.array_equal(ref_votes, g["ref_votes"].astype(np.int64))  # oracle == unmodified reference
    frac = parity.assert_votes_match(votes[valid], ref_votes, nties)
    keep_gpu = votes[valid] < thr
    clean = nties == 0
    assert np.array_equal(keep_gpu[clean], g["ref_keep"][clean])
    assert (keep_gpu != g["ref_keep"]).sum() <= (~clean).sum()
    # bbox of kept points (float32 positions)
    kept = xyz[valid][keep_gpu]
    assert np.array_equal(bbox[:3], kept.min(0)) and np.array_equal(bbox[3:], kept.max(0))
    print(f"tie fraction {frac:.5f}")


@pytest.mark.parametrize("K,W,H,V", [(4, 160, 120, 9), (3, 131, 77, 5)])
def test_filter_neighbour_table(lib_built, K, W, H, V):
    """K < V with the nearest-views table (N2); odd sizes exercise partial chunks and the unaligned path."""
    sc = make_scene(SceneConfig(n_views=V, width=W, height=H, n_sparse=400, seed=21))
    a = dict(poses=sc.cam_from_world.numpy(), intr=sc.intrinsics.numpy())
    nbr = nearest_views_table(a["poses"], K)
    out = R.densify(sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy(), sc.sparse_xyz.numpy(),
                    sc.sparse_offsets.numpy(), a["poses"], a["intr"], nbr, default_vote_threshold(K),
                    align=R.AlignConfig(adaptive_correspondences=False))
    refined = out["refined"]
    thr = default_vote_threshold(K)
    xyz, votes, _ = _run_filter(refined, sc.normal.numpy(), a["poses"], a["intr"], nbr, thr)
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    _assert_xyz_close(xyz[valid], out["points"])
    ref_votes, nties = parity.votes_with_ties(out["points"], out["normals"], out["src_view"], refined, a["poses"], a["intr"], nbr)
    assert np.array_equal(ref_votes, out["votes"])
    parity.assert_votes_match(votes[valid], ref_votes, nties)
    assert ref_votes.max() >= 1  # floaters are being voted on


def test_filter_stride_and_padding(lib_built):
    """downsample_density > 1 (scripts/test.py:206) and -1 padded neighbour rows."""
    sc = make_scene(SceneConfig(n_views=4, width=96, height=64, n_sparse=300, seed=4))
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, 5)  # V-1 = 3 < 5 -> two -1 columns
    assert (nbr[:, 3:] == -1).all()
    out = R.densify(sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy(), sc.sparse_xyz.numpy(),
                    sc.sparse_offsets.numpy(), poses, intr, nbr, 2, align=R.AlignConfig(adaptive_correspondences=False), stride=3)
    refined = out["refined"]
    xyz, votes, _ = _run_filter(refined, sc.normal.numpy(), poses, intr, nbr, 2, stride=3)
    valid = refined[:, ::3, ::3] > 0
    assert votes.shape == valid.shape and np.array_equal(votes != 255, valid)
    _assert_xyz_close(xyz[valid], out["points"])
    ref_votes, nties = parity.votes_with_ties(out["points"], out["normals"], out["src_view"], refined, poses, intr, nbr)
    parity.assert_votes_match(votes[valid], ref_votes, nties, max_tie_fraction=0.05)


@pytest.mark.parametrize("tau", [None, 0.05], ids=["one_sided", "two_sided"])
def test_filter_bilinear_two_sided(lib_built, tau):
    """N3 (parity unpinned - in-repo definition): bilinear sampling, one-sided and two-sided test, compared with the
    float64 statement BIT FOR BIT away from the stated tie bands (tests/parity.py:pair_ties_bilinear)."""
    sc = make_scene(SceneConfig(n_views=6, width=128, height=96, n_sparse=300, seed=9))
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, 3)
    kw = dict(sample_mode="bilinear") if tau is None else dict(sample_mode="bilinear", two_sided_tau=tau)
    out = R.densify(sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy(), sc.sparse_xyz.numpy(),
                    sc.sparse_offsets.numpy(), poses, intr, nbr, 2, align=R.AlignConfig(adaptive_correspondences=False), **kw)
    refined = out["refined"]
    xyz, votes, _ = _run_filter(refined, sc.normal.numpy(), poses, intr, nbr, 2, **kw)
    valid = refined > 0
    assert np.array_equal(votes != 255, valid)
    ref_votes, nties = parity.votes_with_ties(out["points"], out["normals"], out["src_view"], refined, poses, intr, nbr,
                                              sample_mode="bilinear", two_sided_tau=tau)
    assert np.array_equal(ref_votes, out["votes"])  # the tie analysis reproduces the statement's own votes
    frac = parity.assert_votes_match(votes[valid], ref_votes, nties, max_tie_fraction=0.08)
    assert out["votes"].max() >= 1 and frac < 0.08


def test_align_matches_reference_refiner_golden(lib_built, golden_dir):
    """Stage 1 against DepthRefiner.refine_depth run by the reference itself (CPU float32)."""
    from depthdensifier_b200 import ops

    g = np.load(golden_dir / "ref_refiner_cases.npz")
    specs = {
        "default_hashperm": (dict(), True),
        "no_subsample": (dict(adaptive_correspondences=False), True),
        "skip_smoothing": (dict(adaptive_correspondences=False, skip_smoothing=True), True),
        "not_robust": (dict(adaptive_correspondences=False, robust=False), True),
        "mask_none": (dict(adaptive_correspondences=False), False),
        "too_few": (dict(min_correspondences=5000), True),
        "wide_margin": (dict(adaptive_correspondences=False, edge_margin=30, outlier_threshold=1.0), True),
    }
    V = 3
    depth = _cuda(g["mono_depth"])
    pose = _cuda(g["cam_from_world"])
    kmat = _cuda(np.stack([R.kmatrix(i) for i in g["intrinsics"]]))
    sparse = _cuda(g["sparse_xyz"])
    off = _cuda(g["sparse_offsets"])
    maxc = int(np.diff(g["sparse_offsets"]).max())
    for name, (kw, use_mask) in specs.items():
        mask = _cuda(g["mask"]) if use_mask else None
        refined, stats = ops.align_views(depth, mask, pose, kmat, sparse, off, maxc, ops.AlignOptions(**kw))
        torch.cuda.synchronize()
        st = ops.decode_stats(stats)
        refined = refined.cpu().numpy()
        for v in range(V):
            ref = g[f"{name}/{v}/refined"]
            assert st[v]["num_correspondences"] == int(g[f"{name}/{v}/num"]), (name, v, st[v])
            if name == "too_few":
                assert st[v]["status"] == 3
                assert np.array_equal(refined[v], g["mono_depth"][v])  # reference returns the input unchanged
                continue
            assert st[v]["status"] == 0
            assert st[v]["outliers_removed"] == int(g[f"{name}/{v}/removed"]), (name, v)
            assert abs(st[v]["scale_factor"] - float(g[f"{name}/{v}/scale"])) <= 2e-6 * float(g[f"{name}/{v}/scale"])
            assert np.array_equal(refined[v] == 0, ref == 0), (name, v)
            np.testing.assert_allclose(refined[v], ref, rtol=RTOL, atol=0, err_msg=f"{name}/{v}")


def test_align_affine_mode(lib_built):
    """N1 (parity unpinned): scale/shift least squares vs the numpy definition."""
    from depthdensifier_b200 import ops

    sc = make_scene(SceneConfig(n_views=4, width=128, height=96, n_sparse=600, seed=13))
    kmat = np.stack([R.kmatrix(i) for i in sc.intrinsics.numpy()])
    maxc = int(np.diff(sc.sparse_offsets.numpy()).max())
    refined, stats = ops.align_views(sc.mono_depth.cuda(), sc.mask.cuda(), sc.cam_from_world.cuda(), _cuda(kmat),
                                     sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), maxc, ops.AlignOptions(align_mode="affine"))
    st = ops.decode_stats(stats)
    refined = refined.cpu().numpy()
    off = sc.sparse_offsets.numpy()
    for v in range(4):
        r = R.refine_view(sc.mono_depth[v].numpy().copy(), sc.sparse_xyz[off[v]:off[v + 1]].numpy(), sc.cam_from_world[v].numpy(),
                          kmat[v], sc.mask[v].numpy(), R.AlignConfig(align_mode="affine"))
        assert st[v]["status"] == 0 and st[v]["num_correspondences"] == r["num_correspondences"]
        np.testing.assert_allclose(refined[v], r["refined_depth"], rtol=2e-5, atol=0)


def test_depth_refiner_dropin(lib_built, golden_dir):
    """The reference-facing class: same call, same dictionary (depth_refiner.py:207-328)."""
    from depthdensifier_b200 import DepthRefiner, RefinerConfig

    g = np.load(golden_dir / "ref_refiner_cases.npz")
    lo, hi = int(g["sparse_offsets"][1]), int(g["sparse_offsets"][2])
    ref = DepthRefiner(RefinerConfig(verbose=0), adaptive_correspondences=False)
    res = ref.refine_depth(depth_map=g["mono_depth"][1].copy(), normal_map=g["normal"][1], points3D=g["sparse_xyz"][lo:hi],
                           cam_from_world=g["cam_from_world"][1], K=R.kmatrix(g["intrinsics"][1]), mask=g["mask"][1])
    assert set(res) == {"refined_depth", "num_correspondences", "outliers_removed", "scale_factor"}
    assert res["refined_depth"].dtype == np.float32 and res["num_correspondences"] == int(g["no_subsample/1/num"])
    np.testing.assert_allclose(res["refined_depth"], g["no_subsample/1/refined"], rtol=RTOL)
    d_in = g["mono_depth"][1].copy()
    res2 = DepthRefiner(min_correspondences=5000).refine_depth(d_in, None, g["sparse_xyz"][lo:hi], g["cam_from_world"][1],
                                                               R.kmatrix(g["intrinsics"][1]), g["mask"][1])
    assert res2["refined_depth"] is d_in and res2["scale_factor"] == 1.0 and "outliers_removed" not in res2
    res3 = DepthRefiner().refine_depth(d_in, None, np.zeros((0, 3)), g["cam_from_world"][1], R.kmatrix(g["intrinsics"][1]))
    assert res3["num_correspondences"] == 0 and res3["refined_depth"] is d_in


@pytest.mark.parametrize("n,voxel,spread,row_len", [(20000, 0.05, 1.0, 0), (200000, 0.01, 3.0, 37), (1, 0.01, 1.0, 8),
                                                    (5000, 0.001, 40.0, 0), (70001, 0.2, 2.0, 512), (33333, 0.02, 0.3, 33333),
                                                    (200000, 0.001, 40.0, 37)])
def test_voxel_fuse_vs_oracle(lib_built, n, voxel, spread, row_len):
    """N4: keys and counts bit-exact, positions within 1e-5 relative, colours exact.  The 0.001 / 40 cases
    have a grid of more than 2^35 cells and take the hashed path (200 000 points: several sort CTAs and the tiled
    insert), the others the dense-rank path; row_len (the image-width locality hint) must not change the result."""
    from depthdensifier_b200 import ops

    rng = np.random.default_rng(n)
    xyz = (rng.normal(0, spread / 3, (n, 3))).astype(np.float32)
    rgb = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    votes = rng.integers(0, 4, n).astype(np.uint8)
    votes[rng.random(n) < 0.1] = 255
    thr = 2
    sel = votes < thr
    if not sel.any():
        votes[0] = 0
        sel = votes < thr
    origin = R.voxel_origin(xyz[sel], voxel)
    k_ref, m_ref, c_ref, n_ref = R.voxel_fuse(xyz[sel], rgb[sel], voxel, origin)
    grid = ops.make_grid(xyz[sel].min(0), xyz[sel].max(0), voxel)
    assert np.array_equal(np.array(list(grid.origin), np.float32), origin)
    k, m, c, cnt, counts = ops.voxel_fuse(_cuda(xyz), _cuda(rgb), _cuda(votes), thr, grid, row_len=row_len)
    assert counts.cpu().tolist() == [int(sel.sum()), len(k_ref)]
    assert np.array_equal(k.cpu().numpy().view(np.uint64), k_ref)
    assert np.array_equal(cnt.cpu().numpy(), n_ref)
    assert np.array_equal(c.cpu().numpy(), c_ref)
    err = np.abs(m.cpu().numpy().astype(np.float64) - m_ref).max()
    assert err <= RTOL * max(1.0, np.abs(m_ref).max())
    keys_all = ops.voxel_keys(_cuda(xyz[sel]), voxel, origin).cpu().numpy().view(np.uint64)
    assert np.array_equal(keys_all, R.voxel_keys(xyz[sel], voxel, origin))


def test_pipeline_end_to_end_vs_oracle(lib_built):
    """align -> back-project+vote -> fuse on a scene with an unrefinable view, against the oracle chain."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.engine import DensifyConfig, DensifyEngine

    sc = make_scene(SceneConfig(n_views=8, width=144, height=104, n_sparse=900, seed=17))
    K = 4
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, K)
    thr = default_vote_threshold(K)
    out = R.densify(sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy(), sc.sparse_xyz.numpy(),
                    sc.sparse_offsets.numpy(), poses, intr, nbr, thr, randperm=lambda n: hash_perm(n, 0), voxel=0.02)
    eng = DensifyEngine(DensifyConfig(voxel=0.02))
    res = eng.run(sc.mono_depth.cuda(), sc.normal.cuda(), sc.mask.cuda(), sc.rgb.cuda(), sc.cam_from_world.cuda(),
                  sc.intrinsics.cuda(), sc.sparse_xyz.cuda(), sc.sparse_offsets.cuda(), _cuda(nbr.astype(np.int32)))
    torch.cuda.synchronize()
    refined = res.refined.cpu().numpy()
    np.testing.assert_allclose(refined, out["refined"], rtol=RTOL, atol=0)
    valid = out["refined"] > 0
    votes = res.votes.cpu().numpy()
    assert np.array_equal(votes != 255, valid)
    _assert_xyz_close(res.xyz.cpu().numpy()[valid], out["points"])
    # votes: computed by the GPU from ITS refined depth (<=1e-5 off the oracle's) -> compare keep counts loosely,
    # the exact comparison on identical inputs is test_filter_*.
    keep_gpu = votes[valid] < thr
    assert abs(int(keep_gpu.sum()) - int(out["keep"].sum())) <= 0.002 * len(keep_gpu)
    assert (keep_gpu != out["keep"]).mean() < 0.002
    # fusion of the GPU's own kept points must equal the oracle fusion of those same points
    xyz_kept = res.xyz.cpu().numpy()[valid][keep_gpu]
    rgb_kept = sc.rgb.numpy()[valid][keep_gpu]
    origin = np.array(list(res.host_grid().origin), np.float32)  # derived on the device from the alignment kernel's box
    assert (origin <= xyz_kept.min(0)).all()
    k_ref, m_ref, c_ref, n_ref = R.voxel_fuse(xyz_kept, rgb_kept, 0.02, origin)
    assert res.counts.cpu().tolist() == [len(xyz_kept), len(k_ref)]
    assert np.array_equal(res.voxel_keys.cpu().numpy().view(np.uint64), k_ref)
    assert np.array_equal(res.voxel_count.cpu().numpy(), n_ref)
    assert np.array_equal(res.voxel_rgb.cpu().numpy(), c_ref)
    assert np.abs(res.voxel_xyz.cpu().numpy() - m_ref).max() <= RTOL * max(1.0, np.abs(m_ref).max())


def test_voxel_partials_and_merge_bit_exact(lib_built):
    """Multi-GPU form of N4: partial sums and their merge are integer arithmetic -> bit-exact against the
    numpy statement in tests/cpu_backend.py, and merge(partials of two halves) == fuse(all), also when the
    records arrive in random order."""
    _check_partials_and_merge(far=False)


def test_voxel_partials_and_merge_bit_exact_over_2e35_cells(lib_built):
    """The same on a grid of more than 2^35 cells (a second cluster 400 m away): the hashed path, no ownership tiles."""
    _check_partials_and_merge(far=True)


def _check_partials_and_merge(far: bool):
    from cpu_backend import finalize_numpy, merge_numpy, pack_records, partial_sums_numpy, unpack_records
    from depthdensifier_b200 import ops

    rng = np.random.default_rng(5)
    n = 150000
    xyz = rng.normal(0, 0.7, (n, 3)).astype(np.float32)
    if far:
        xyz[rng.random(n) < 0.2] += np.float32(400.0)
    rgb = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    voxel = 0.02
    grid = ops.make_grid(xyz.min(0), xyz.max(0), voxel)
    origin = np.array(list(grid.origin), np.float32)
    uk, sums, csum, cnt = partial_sums_numpy(xyz, rgb, np.float32(voxel), origin)
    rec, counts = ops.voxel_fuse_partial(_cuda(xyz), _cuda(rgb), None, 1, grid, row_len=300)
    mv = int(counts[1])
    assert counts.cpu().tolist() == [n, len(uk)]
    assert np.array_equal(rec[:mv].cpu().numpy(), pack_records(uk, sums, csum, cnt))
    pk, ps, pr, pc = unpack_records(rec[:mv].cpu().numpy())
    assert np.array_equal(pk, uk) and np.array_equal(ps, sums) and np.array_equal(pr, csum) and np.array_equal(pc, cnt)
    # split the points in two "ranks", fuse partially, merge the concatenated records
    h = n // 3
    parts = [ops.voxel_fuse_partial(_cuda(xyz[a:b]), _cuda(rgb[a:b]), None, 1, grid) for a, b in ((0, h), (h, n))]
    cat = torch.cat([p[0][: int(p[1][1])] for p in parts]).contiguous()
    k, x, c, m, mc = ops.voxel_merge_partials(cat, grid, trim=True)
    assert mc.cpu().tolist() == [cat.shape[0], len(uk)]
    perm = torch.from_numpy(rng.permutation(cat.shape[0])).cuda()
    shuffled = ops.voxel_merge_partials(cat[perm].contiguous(), grid, trim=True)
    for i in range(5):
        assert np.array_equal(shuffled[i].cpu().numpy(), (k, x, c, m, mc)[i].cpu().numpy())
    # ownership tiles (none on a grid beyond 2^35 cells): the prefix of records per tile, and merges restricted to
    # tile ranges
    from cpu_backend import OracleBackend

    n_tiles, cells_per_tile = ops.fuse_tile_info(grid)
    if far:
        assert n_tiles == 0
    else:
        assert (n_tiles, cells_per_tile) == OracleBackend().fuse_tile_info(grid)
        tp = torch.full((n_tiles + 1,), -7, dtype=torch.int32, device="cuda")
        rec2, _ = ops.voxel_fuse_partial(_cuda(xyz), _cuda(rgb), None, 1, grid, tile_prefix=tp)
        tiles_of = OracleBackend()._tile_of_keys(uk, grid)
        assert np.array_equal(tp.cpu().numpy(), np.searchsorted(tiles_of, np.arange(n_tiles + 1)))
        cut = int(np.searchsorted(np.cumsum(np.bincount(tiles_of, minlength=n_tiles)), len(uk) // 2))
        halves = [ops.voxel_merge_partials(cat, grid, trim=True, tile_range=r) for r in ((0, cut), (cut, n_tiles))]
        assert len(halves[0][0]) > 0 and len(halves[1][0]) > 0
        for i in range(4):
            assert np.array_equal(torch.cat([halves[0][i], halves[1][i]]).cpu().numpy(), (k, x, c, m)[i].cpu().numpy())
    full = ops.voxel_fuse(_cuda(xyz), _cuda(rgb), None, 1, grid)
    assert np.array_equal(k.cpu().numpy(), full[0].cpu().numpy()) and np.array_equal(m.cpu().numpy(), full[3].cpu().numpy())
    assert np.array_equal(x.cpu().numpy(), full[1].cpu().numpy()) and np.array_equal(c.cpu().numpy(), full[2].cpu().numpy())
    ref_xyz, ref_rgb = finalize_numpy(uk, sums, csum, cnt, np.float32(voxel), origin)
    assert np.array_equal(x.cpu().numpy(), ref_xyz) and np.array_equal(c.cpu().numpy(), ref_rgb)
    mk, ms, mcs, mn = merge_numpy(uk, sums, csum, cnt)
    assert np.array_equal(mk, uk) and np.array_equal(mn, cnt)


@pytest.mark.parametrize("in_place", [True, False])
def test_run_host_matches_device_pipeline(lib_built, in_place):
    """The pipelined host entry point (chunked uploads overlapped with alignment, normals read in place from
    pinned host memory or copied) returns exactly what the device-resident pipeline computes."""
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig

    sc = make_scene(SceneConfig(n_views=7, width=150, height=96, n_sparse=700, seed=3))
    K = 4
    nbr = nearest_views_table(sc.cam_from_world.numpy(), K)
    sd = ShardedDensifier(DensifyConfig(voxel=0.02), torch.device("cuda", 0), 0, 1, 7, 0, 7, sc.cam_from_world, sc.intrinsics,
                          nbr, 96, 150)
    host = (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets)
    res = sd.run(*[t.cuda() for t in host])
    mv = int(res.counts[1])
    pinned = sd.pin_host_inputs(*host, pack_mask=in_place)  # the bit-packed mask in one of the two variants
    for _ in range(2):  # second call reuses the staging buffers
        out = sd.run_host(*pinned, normals_in_place=in_place, chunk_views=3)
    assert out["num_points"] == int(res.counts[0]) and len(out["keys"]) == mv
    assert np.array_equal(out["keys"].numpy(), res.voxel_keys[:mv].cpu().numpy())
    assert np.array_equal(out["xyz"].numpy(), res.voxel_xyz[:mv].cpu().numpy())
    assert np.array_equal(out["rgb"].numpy(), res.voxel_rgb[:mv].cpu().numpy())
    assert np.array_equal(out["count"].numpy(), res.voxel_count[:mv].cpu().numpy())
    expected_h2d = sum(t.numel() * t.element_size() for i, t in enumerate(pinned) if not (in_place and i == 1))
    assert out["h2d_bytes"] == expected_h2d
    # the two halves, pipelined: three scenes in flight (the third is submitted before the first is collected)
    tickets = [sd.submit_host(*pinned, normals_in_place=in_place, chunk_views=4) for _ in range(2)]
    outs = [sd.collect_host(tickets[0])]
    tickets.append(sd.submit_host(*pinned, normals_in_place=in_place, chunk_views=2))
    outs += [sd.collect_host(tickets[1]), sd.collect_host(tickets[2])]
    for o in outs[1:]:  # (outs[0] shares its pinned buffers with the third call)
        assert o["num_points"] == int(res.counts[0]) and np.array_equal(o["keys"].numpy(), res.voxel_keys[:mv].cpu().numpy())
        assert np.array_equal(o["xyz"].numpy(), res.voxel_xyz[:mv].cpu().numpy())
        assert np.array_equal(o["rgb"].numpy(), res.voxel_rgb[:mv].cpu().numpy())
        assert np.array_equal(o["count"].numpy(), res.voxel_count[:mv].cpu().numpy())
