"""GPU tests of the hashed multi-GPU fusion (include/ddn_b200.h: ddn_fuse_finish_hashed_partial, ddn_fuse_merge_hashed_peers)
driven with VIRTUAL ranks on one GPU: R sessions and hash buffers in one process, whose local addresses stand in for the
peers' NVLink mappings, so the exchange logic is under bit-exact test on a one-GPU box.  The rank-ordered concatenation
of the owners' voxels must equal the one-GPU hashed result, and on grids the dense path can hold, the dense result."""

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from hashed_plan import share_bound, splitters
from test_gpu_hashed_fuse import CLOUDS, DOME, DOME_VOXEL, _assert_oracle_voxels, _box, _cuda, _engine, _scene_args

pytestmark = pytest.mark.gpu

S = 4096


def _deal(n, R, skew=None):
    """Contiguous blocks of [0, n) for R ranks; ``skew``: explicit fractions of the points per rank."""
    if skew is None:
        b = np.linspace(0, n, R + 1).astype(int)
        b[1] = max(b[1] // 5, 0)  # uneven shares
    else:
        b = np.concatenate([[0], np.cumsum(np.asarray(skew) * n)]).astype(int)
        b[-1] = n
    return [(int(b[r]), int(b[r + 1])) for r in range(R)]


class VirtualRanks:
    """R ranks in one process: a session, hash buffers, records and samples each."""

    def __init__(self, R, n_max, max_cells=1 << 20, n_dedup=0):
        from depthdensifier_b200 import ops

        self.R = R
        # output capacity of both merges, as ShardedDensifier sizes it
        self.cap = max(ops.hashed_merge_capacity(max(n_max, 1), R), n_max + 24576 * R + 1024)
        self.sessions = [ops.FuseSession("cuda", max_cells=max_cells, tile_prefix=True) for _ in range(R)]
        self.hfs = [ops.HashFuse("cuda", max(n_max + n_dedup, self.cap)) for _ in range(R)]
        self.records = [torch.empty((max(n_max, 1), 6), dtype=torch.int64, device="cuda") for _ in range(R)]
        self.samples = [ops.new_hash_samples("cuda") for _ in range(R)]
        self.plans = [torch.zeros(64, dtype=torch.int64, device="cuda") for _ in range(R)]

    def step(self, parts, thr, begin, mode=0, dedup=None):
        """One step as ShardedDensifier enqueues it: dense partial, hashed partial, then dense merge, hashed merge on the
        same outputs (mode 0); mode 1 (the hashed path forced on an OK grid) enqueues only the hashed halves.  ``parts``:
        per rank (xyz, rgb, votes) CUDA tensors.  Returns the concatenated outputs, the per-rank counts after the partial
        and after the merge, and the plans."""
        from depthdensifier_b200 import ops

        R = self.R
        dense = mode == 0
        part_counts = []
        for r, (x, c, v) in enumerate(parts):
            sess = self.sessions[r]
            begin(sess)
            if dense:
                sess.mark_points(x, v, thr)
                ops.fuse_finish_partial(sess, x, c, v, thr, self.records[r])
            ops.fuse_finish_hashed_partial(sess, self.hfs[r], x, c, v, thr, self.records[r], self.samples[r], dedup_xyz=dedup, mode=mode)
            part_counts.append(sess.counts.clone())
        pr = [t.data_ptr() for t in self.records]
        ps = [t.data_ptr() for t in self.samples]
        pp = [s.tile_prefix.data_ptr() for s in self.sessions]
        outs, counts = [], []
        for r in range(R):
            sess, hf = self.sessions[r], self.hfs[r]
            out = ops.new_voxel_outputs(self.cap, "cuda")
            if dense:
                out = ops.fuse_merge_peers(sess, r, R, pr, pp, self.plans[r], self.cap, out=out, drop_xyz=dedup)[:4]
            k, x, c, n, cnt = ops.fuse_merge_hashed_peers(sess, hf, r, R, pr, ps, self.plans[r], self.cap, out=out)
            mv = int(cnt[1])
            outs.append((k[:mv].clone(), x[:mv].clone(), c[:mv].clone(), n[:mv].clone()))
            counts.append(cnt.cpu().tolist())
        for hf in self.hfs:
            hf.check()
        cat = [torch.cat([o[i] for o in outs]) for i in range(4)]
        return cat, [c.cpu().tolist() for c in part_counts], counts, [p.cpu().tolist() for p in self.plans]

    def host_records(self, parts_counts):
        return [self.records[r][: parts_counts[r][1], 0].cpu().numpy().view(np.uint64) for r in range(self.R)]


def _same(cat, ref, mv=None):
    for a, b in zip(cat, ref[:4]):
        b = b if mv is None else b[:mv]
        assert a.shape == b.shape and torch.equal(a, b)


def _check_plans(vr, part_counts, plans, counts):
    """The plans follow the numpy statement (tests/hashed_plan.py): the same splitters, shares that add up to all
    records, every share within the bound."""
    recs = vr.host_records(part_counts)
    total = sum(len(k) for k in recs)
    ks = splitters(recs, S)
    for r, p in enumerate(plans):
        assert np.uint64(p[0] % 2**64) == ks[r] and np.uint64(p[1] % 2**64) == ks[r + 1]
        assert p[3] == total and p[2] <= share_bound(total, vr.R, S) and p[2] <= vr.cap
        assert counts[r][1] <= p[2]
    assert sum(p[2] for p in plans) == total
    return total


def _one_gpu(xyz, rgb, votes, thr, begin, dedup=None):
    from depthdensifier_b200 import ops

    sess = ops.FuseSession("cuda", max_cells=1 << 34)
    begin(sess)
    sess.mark_points(xyz, votes, thr)
    if dedup is not None:
        sess.unmark_points(dedup)
    dense = [t.clone() for t in ops.fuse_finish(sess, xyz, rgb, votes, thr)]
    hf = ops.HashFuse("cuda", max(xyz.shape[0] + (0 if dedup is None else dedup.shape[0]), 1))
    hashed = ops.fuse_finish_hashed(sess, hf, xyz, rgb, votes, thr, dedup_xyz=dedup, mode=1)
    mv = int(hashed[4][1])
    return [t[:mv].clone() for t in hashed[:4]], hashed[4].cpu().tolist(), [t[:mv] for t in dense[:4]], dense[4].cpu().tolist()


def _cloud_inputs(case):
    xyz, votes, thr, voxel = CLOUDS[case]
    n = len(xyz)
    rgb = np.random.default_rng(n).integers(0, 256, (n, 3)).astype(np.uint8)
    lo = xyz.min(0) - 0.013 if n else np.zeros(3, np.float32)
    hi = xyz.max(0) + 0.021 if n else np.ones(3, np.float32)
    box = _box(lo, hi)
    return _cuda(xyz), _cuda(rgb), _cuda(votes), thr, (lambda sess: sess.begin([box], voxel))


def _parts(d, bounds):
    return [tuple(t[a:b] for t in d) for a, b in bounds]


@pytest.mark.parametrize("R", [2, 3, 8, 16])
@pytest.mark.parametrize("case", ["threshold_drops", "one_voxel", "many_voxels"])
def test_virtual_ranks_equal_one_gpu(lib_built, case, R):
    """A grid too large for the virtual ranks' sessions (both forms enqueued): the owners' voxels in rank order ==
    one-GPU hashed == dense on the same grid in a session that holds it; the ranks' point counts add up to the one-GPU
    count; the plans follow the numpy statement of the splitter rule."""
    x, c, v, thr, begin = _cloud_inputs(case)
    bounds = _deal(x.shape[0], R)
    vr = VirtualRanks(R, max(b - a for a, b in bounds))
    cat, part_counts, counts, plans = vr.step(_parts((x, c, v), bounds), thr, begin)
    hashed, hcounts, dense, dcounts = _one_gpu(x, c, v, thr, begin)
    assert hcounts == dcounts
    _same(cat, hashed)
    _same(cat, dense)
    assert sum(p[0] for p in part_counts) == hcounts[0]
    assert _check_plans(vr, part_counts, plans, counts) >= hcounts[1]
    assert bool((cat[0][1:] > cat[0][:-1]).all())


@pytest.mark.parametrize("skew", ["one_empty_one_full", "empty_ranks", "one_rank"])
def test_skewed_shares(lib_built, skew):
    """One rank with no points and one with nearly all; ranks without views (shard_bounds at small V); one rank."""
    x, c, v, thr, begin = _cloud_inputs("many_voxels")
    n = x.shape[0]
    R, frac = {"one_empty_one_full": (4, [0.0, 0.97, 0.02, 0.01]), "empty_ranks": (8, [0.3, 0.3, 0.4, 0, 0, 0, 0, 0]),
               "one_rank": (1, [1.0])}[skew]
    bounds = _deal(n, R, frac)
    vr = VirtualRanks(R, max(b - a for a, b in bounds))
    cat, part_counts, counts, plans = vr.step(_parts((x, c, v), bounds), thr, begin)
    hashed, hcounts, _, _ = _one_gpu(x, c, v, thr, begin)
    _same(cat, hashed)
    _check_plans(vr, part_counts, plans, counts)


def test_one_voxel_on_every_rank_and_straddling_keys(lib_built):
    """Every rank holds the same voxel (R records of one key), and runs of consecutive keys that every rank holds lie
    across the splitters."""
    R = 8
    rng = np.random.default_rng(3)
    voxel = 0.01
    line = (np.arange(60000, dtype=np.float32)[:, None] * np.float32(voxel) + 0.005) * np.array([[1, 0, 0]], np.float32)
    xyz = np.concatenate([np.tile(line, (R, 1)), np.full((R * 100, 3), 0.3051, np.float32)])
    xyz = xyz[rng.permutation(len(xyz))]  # every rank gets a share of every key
    rgb = rng.integers(0, 256, (len(xyz), 3)).astype(np.uint8)
    votes = np.zeros(len(xyz), np.uint8)
    d = (_cuda(xyz), _cuda(rgb), _cuda(votes))
    box = _box(xyz.min(0) - 0.01, xyz.max(0) + 0.01)
    begin = lambda sess: sess.begin([box], voxel)
    bounds = _deal(len(xyz), R, [1 / R] * R)
    vr = VirtualRanks(R, max(b - a for a, b in bounds))
    cat, part_counts, counts, plans = vr.step(_parts(d, bounds), 1, begin)
    hashed, hcounts, _, _ = _one_gpu(*d, 1, begin)
    _same(cat, hashed)
    _check_plans(vr, part_counts, plans, counts)
    assert int(cat[3].max()) >= R * 100


def test_adversarial_samples(lib_built):
    """Rank 0 holds one voxel per z-layer, so its consecutive samples are two layers apart; rank 1 puts 300000 voxels
    into the one layer between two of them.  The shares still stay within the bound."""
    R, voxel = 4, 0.01
    coarse = np.full((8192, 3), 0.5 * voxel, np.float32)
    coarse[:, 2] = (np.arange(8192) + 0.5) * voxel
    i = np.arange(300000)
    fine = np.stack([(i % 548 + 0.5) * voxel, (i // 548 + 0.5) * voxel, np.full(len(i), 2001.5 * voxel)], 1).astype(np.float32)
    xyz = np.concatenate([coarse, fine, fine[::300], coarse[::5]])
    rgb = np.random.default_rng(1).integers(0, 256, (len(xyz), 3)).astype(np.uint8)
    d = (_cuda(xyz), _cuda(rgb), _cuda(np.zeros(len(xyz), np.uint8)))
    box = _box(xyz.min(0) - voxel, xyz.max(0) + voxel)
    begin = lambda sess: sess.begin([box], voxel)
    n0, n1, n2 = len(coarse), len(fine), len(fine[::300])
    bounds = [(0, n0), (n0, n0 + n1), (n0 + n1, n0 + n1 + n2), (n0 + n1 + n2, len(xyz))]
    vr = VirtualRanks(R, max(b - a for a, b in bounds))
    cat, part_counts, counts, plans = vr.step(_parts(d, bounds), 1, begin)
    hashed, _, _, _ = _one_gpu(*d, 1, begin)
    _same(cat, hashed)
    _check_plans(vr, part_counts, plans, counts)


@pytest.mark.parametrize("R", [2, 8])
def test_dome_scene_too_large_grid(lib_built, R):
    """The dome scene's kept points on a TOO_LARGE grid (mode 0, dense kernels enqueued too): the one-GPU engine's voxels
    bit for bit, and the oracle's."""
    from depthdensifier_b200 import _lib

    sc = make_scene(SceneConfig(**DOME))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    res = _engine(voxel=DOME_VOXEL).run(*_scene_args(sc, nbr))
    assert res.session.grid_state().status == _lib.GRID_HASHED
    flat = (res.xyz.view(-1, 3), res.grid_rgb().reshape(-1, 3).contiguous(), res.votes.view(-1))
    per_view = res.xyz.shape[1] * res.xyz.shape[2]
    views = [(a * per_view, b * per_view) for a, b in _view_bounds(res.xyz.shape[0], R)]
    vr = VirtualRanks(R, max(b - a for a, b in views))
    begin = lambda sess: sess.begin([res.bbox_valid], DOME_VOXEL)
    cat, part_counts, counts, plans = vr.step(_parts(flat, views), res.vote_threshold, begin, mode=0)
    assert all(s.grid_state().status == _lib.GRID_HASHED for s in vr.sessions)
    _same(cat, (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count))
    assert sum(p[0] for p in part_counts) == int(res.counts[0])
    _check_plans(vr, part_counts, plans, counts)
    kx, krgb = res.kept_points()
    _assert_oracle_voxels(*(t.cpu().numpy() for t in cat), kx.cpu().numpy(), krgb.cpu().numpy(), DOME_VOXEL, list(res.host_grid().origin))


def _view_bounds(V, R):
    from depthdensifier_b200.distributed import shard_bounds

    return shard_bounds(V, R)


def test_flag_when_only_the_sum_reaches_2_24(lib_built):
    """A voxel that holds fewer than 2^24 points on every rank but 2^24 or more in all: the owner reports it."""
    R = 2
    n = (1 << 23) + 4096
    xyz = np.full((2 * n, 3), 0.5, np.float32)
    xyz[-8:] = 3.0  # a second voxel, owned by the other rank
    d = (_cuda(xyz), torch.zeros((2 * n, 3), dtype=torch.uint8, device="cuda"), torch.zeros(2 * n, dtype=torch.uint8, device="cuda"))
    box = _box(np.zeros(3, np.float32), np.full(3, 4.0, np.float32))
    vr = VirtualRanks(R, n)
    cat, part_counts, counts, plans = vr.step(_parts(d, [(0, n), (n, 2 * n)]), 1, lambda s: s.begin([box], 1.0), mode=1)
    assert all(p[0] == n for p in part_counts)
    assert int(cat[3][0]) == 2 * n - 8 and int(cat[3][1]) == 8
    assert sorted(c[0] for c in counts) == [-1, n]


@pytest.mark.parametrize("R", [3, 8])
def test_dedup_n5(lib_built, R):
    """N5: every rank tombstones all ranks' sparse points; the result equals the one-GPU hashed result with the same
    points and, on an OK grid, the dense result with the cells unmarked (merge_sparse(dedup=True), tested there)."""
    x, c, v, thr, begin = _cloud_inputs("threshold_drops")
    dedup = x[::37].contiguous()
    bounds = _deal(x.shape[0], R)
    vr = VirtualRanks(R, max(b - a for a, b in bounds), max_cells=1 << 34, n_dedup=dedup.shape[0])
    cat, part_counts, counts, plans = vr.step(_parts((x, c, v), bounds), thr, begin, mode=1, dedup=dedup)
    assert all(s.grid_state().status == 0 for s in vr.sessions)
    hashed, hcounts, dense, dcounts = _one_gpu(x, c, v, thr, begin, dedup=dedup)
    assert hcounts == dcounts and hcounts[1] > 0
    _same(cat, hashed)
    _same(cat, dense)
    assert sum(p[0] for p in part_counts) == hcounts[0]


def test_dense_hashed_hashed_dense_steps(lib_built):
    """dense, hashed, hashed, dense on the same virtual ranks (both forms enqueued, mode 0): every step equals the one-GPU
    engine's fusion of the same kept points, and the tables are empty afterwards."""
    from depthdensifier_b200 import _lib, ops

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    args = _scene_args(sc, nbr)
    R = 3
    vr = None
    for voxel, status in [(0.05, _lib.GRID_OK), (0.02, _lib.GRID_HASHED), (0.015, _lib.GRID_HASHED), (0.05, _lib.GRID_OK)]:
        res = _engine(max_cells=1 << 26, voxel=voxel).run(*args)
        assert res.session.grid_state().status == status
        flat = (res.xyz.view(-1, 3), res.grid_rgb().reshape(-1, 3).contiguous(), res.votes.view(-1))
        per_view = res.xyz.shape[1] * res.xyz.shape[2]
        views = [(a * per_view, b * per_view) for a, b in _view_bounds(res.xyz.shape[0], R)]
        if vr is None:
            vr = VirtualRanks(R, max(b - a for a, b in views), max_cells=1 << 26)
        parts = _parts(flat, views)

        def begin(sess, box=res.bbox_valid, voxel=voxel):
            sess.begin([box], voxel)

        cat, part_counts, counts, plans = vr.step(parts, res.vote_threshold, begin, mode=0)
        assert all(s.grid_state().status == status for s in vr.sessions)
        assert all(hf.ran() == (status == _lib.GRID_HASHED) for hf in vr.hfs)
        _same(cat, (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count))
    for hf in vr.hfs:
        assert bool((hf.table == 255).all()) and bool((hf.slots[: hf.cap_voxels * 4] == 255).all())


@pytest.mark.parametrize("dedup", [False, True])
def test_sharded_one_rank_equals_engine_on_dome(lib_built, dedup):
    """ShardedDensifier with world == 1 fuses the dome scene (its grid exceeds the session's bitmap) as DensifyEngine.run
    does, bit for bit, through run and through run_host."""
    from depthdensifier_b200 import _lib, ops
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig

    sc = make_scene(SceneConfig(**DOME))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    V, H, W = sc.mono_depth.shape
    cfg = DensifyConfig(voxel=DOME_VOXEL, dedup_sparse=dedup,
                        align=ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True))
    ref = _engine(voxel=DOME_VOXEL, dedup_sparse=dedup).run(*_scene_args(sc, nbr))
    assert ref.session.grid_state().status == _lib.GRID_HASHED
    sd = ShardedDensifier(cfg, "cuda", 0, 1, V, 0, V, sc.cam_from_world, sc.intrinsics, nbr, H, W)
    inputs = tuple(t.cuda().contiguous() for t in (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets))
    res = sd.run(*inputs)
    mv = res.check()
    assert mv == ref.voxel_keys.shape[0] and int(res.counts[0]) == int(ref.counts[0])
    _same((res.voxel_keys[:mv], res.voxel_xyz[:mv], res.voxel_rgb[:mv], res.voxel_count[:mv]), (ref.voxel_keys, ref.voxel_xyz, ref.voxel_rgb, ref.voxel_count))
    host = sd.pin_host_inputs(*(t.contiguous() for t in (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets)))
    out = sd.run_host(*host, chunk_views=4)
    assert out["grid"] is not None and out["num_points"] == int(ref.counts[0])
    for name, t in (("keys", ref.voxel_keys), ("xyz", ref.voxel_xyz), ("rgb", ref.voxel_rgb), ("count", ref.voxel_count)):
        assert np.array_equal(out[name].numpy(), t.cpu().numpy()), name
