"""GPU tests of the multi-GPU fused normals (include/ddn_b200.h: the *_normals forms of ddn_fuse_finish_partial,
ddn_fuse_merge_peers, ddn_fuse_finish_hashed_partial and ddn_fuse_merge_hashed_peers) with VIRTUAL ranks on one GPU, as
tests/test_gpu_hashed_peers.py drives the plain forms.  The rank-ordered concatenation of the owners' voxels, normals
included, must equal the one-GPU normals result bit for bit and the numpy statement of tests/normal_oracle.py; the
80-byte partial records must hold the plain record, the per-rank normal sums and a zero word; and nothing but the
normals may change with the option on."""

import json
import socket
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from depthdensifier_b200.neighbours import nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene

import cpu_backend as CB
import normal_oracle as NO
from test_gpu_hashed_fuse import CLOUDS, DOME, DOME_VOXEL, _box, _cuda, _engine, _scene_args
from test_gpu_hashed_peers import _deal, _parts

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _unit_normals(n, seed):
    """Unit float32 normals with components in [-1, 1], one in 50 zero (a pixel without a finite normal)."""
    rng = np.random.default_rng(seed)
    v = rng.normal(size=(n, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    v[rng.random(n) < 0.02] = 0.0
    return v.astype(np.float32)


class NormalRanks:
    """R ranks in one process, each with a session, hash buffers, records and samples; ``normals`` selects the
    fused-normal forms (80-byte records) or the plain ones."""

    def __init__(self, R, n_max, normals, max_cells=1 << 20, n_dedup=0):
        from depthdensifier_b200 import _lib, ops

        self.R, self.normals = R, normals
        self.cap = max(ops.hashed_merge_capacity(max(n_max, 1), R), n_max + 24576 * R + 1024)
        width = _lib.RECORD_NORMAL_WORDS if normals else _lib.RECORD_WORDS
        self.sessions = [ops.FuseSession("cuda", max_cells=max_cells, tile_prefix=True) for _ in range(R)]
        self.hfs = [ops.HashFuse("cuda", max(n_max + n_dedup, self.cap)) for _ in range(R)]
        self.records = [torch.full((max(n_max, 1), width), -7, dtype=torch.int64, device="cuda") for _ in range(R)]
        self.samples = [ops.new_hash_samples("cuda") for _ in range(R)]
        self.plans = [torch.zeros(64, dtype=torch.int64, device="cuda") for _ in range(R)]

    def step(self, parts, thr, begin, mode=0, dedup=None):
        """ShardedDensifier's order: dense partial, hashed partial, barrier, dense merge, hashed merge on the same outputs
        (mode 1: the hashed halves only).  ``parts``: per rank (xyz, rgb, votes, normal).  Returns the concatenated
        outputs (keys, xyz, rgb, count[, normal]), per-rank counts after the partial and after the merge, and a copy of
        every rank's records."""
        from depthdensifier_b200 import ops

        R, dense = self.R, mode == 0
        part_counts, recs = [], []
        for r, (x, c, v, nrm) in enumerate(parts):
            sess = self.sessions[r]
            kw = {"normal": nrm} if self.normals else {}
            begin(sess)
            if dense:
                sess.mark_points(x, v, thr)
                ops.fuse_finish_partial(sess, x, c, v, thr, self.records[r], **kw)
            ops.fuse_finish_hashed_partial(sess, self.hfs[r], x, c, v, thr, self.records[r], self.samples[r], dedup_xyz=dedup, mode=mode, **kw)
            part_counts.append(sess.counts.clone())
        for r in range(R):
            recs.append(self.records[r][: int(part_counts[r][1])].clone())
        pr = [t.data_ptr() for t in self.records]
        ps = [t.data_ptr() for t in self.samples]
        pp = [s.tile_prefix.data_ptr() for s in self.sessions]
        n_out = 5 if self.normals else 4
        outs, counts = [], []
        for r in range(R):
            sess, hf = self.sessions[r], self.hfs[r]
            out = ops.new_voxel_outputs(self.cap, "cuda", normals=self.normals)
            if dense:
                out = ops.fuse_merge_peers(sess, r, R, pr, pp, self.plans[r], self.cap, out=out, drop_xyz=dedup, normals=self.normals)[:n_out]
            *vox, cnt = ops.fuse_merge_hashed_peers(sess, hf, r, R, pr, ps, self.plans[r], self.cap, out=out, normals=self.normals)
            mv = int(cnt[1])
            outs.append([t[:mv].clone() for t in vox])
            counts.append(cnt.cpu().tolist())
        for hf in self.hfs:
            hf.check()
        cat = [torch.cat([o[i] for o in outs]) for i in range(n_out)]
        return cat, [c.cpu().tolist() for c in part_counts], counts, recs


def _one_gpu(xyz, rgb, votes, nrm, thr, begin, dedup=None):
    """ddn_fuse_finish_normals and ddn_fuse_finish_hashed_normals (mode 1) over all points: (hashed, dense) outputs."""
    from depthdensifier_b200 import ops

    sess = ops.FuseSession("cuda", max_cells=1 << 34)
    begin(sess)
    sess.mark_points(xyz, votes, thr)
    if dedup is not None:
        sess.unmark_points(dedup)
    dense = [t.clone() for t in ops.fuse_finish(sess, xyz, rgb, votes, thr, normal=nrm)]
    grid = sess.host_grid()
    hf = ops.HashFuse("cuda", max(xyz.shape[0] + (0 if dedup is None else dedup.shape[0]), 1))
    hashed = ops.fuse_finish_hashed(sess, hf, xyz, rgb, votes, thr, dedup_xyz=dedup, mode=1, normal=nrm)
    mv = int(hashed[5][1])
    return [t[:mv].clone() for t in hashed[:5]], [t[: int(dense[5][1])] for t in dense[:5]], grid


def _same(cat, ref):
    assert len(cat) == len(ref)
    for a, b in zip(cat, ref):
        assert a.shape == b.shape and torch.equal(a, b)


def _participating(x, v, nrm, thr, grid, dedup=None):
    """Host copies of the points that take part: vote below thr, not in a dedup cell (the grids here enclose every point)."""
    x, v, nrm = x.cpu().numpy(), v.cpu().numpy(), nrm.cpu().numpy()
    voxel, origin = np.float32(grid.voxel), np.array(list(grid.origin), np.float32)
    keep = v < thr
    if dedup is not None:
        _, keys = CB.canonical_keys(x, voxel, origin)
        _, drop = CB.canonical_keys(dedup.cpu().numpy().astype(np.float32), voxel, origin)
        keep &= ~np.isin(keys, drop)
    return x[keep], nrm[keep], voxel, origin


def _assert_oracle(cat, xyz, votes, nrm, thr, grid, dedup=None):
    px, pn, voxel, origin = _participating(xyz, votes, nrm, thr, grid, dedup)
    keys, sums = NO.fused_normal_sums(px, pn, voxel, origin)
    assert np.array_equal(cat[0].cpu().numpy(), keys)
    assert np.array_equal(cat[4].cpu().numpy(), NO.final_normals(sums))


def _assert_records(vr_on, recs_on, recs_off, parts, thr, grid):
    """Words 0-5 of every 80-byte record are the plain record, words 6-8 the rank's numpy normal sums, word 9 zero."""
    for r, (on, off) in enumerate(zip(recs_on, recs_off)):
        assert on.shape[0] == off.shape[0] and on.shape[1] == 10
        assert torch.equal(on[:, :6], off)
        assert bool((on[:, 9] == 0).all())
        x, _, v, nrm = parts[r]
        px, pn, voxel, origin = _participating(x, v, nrm, thr, grid)
        keys, sums = NO.fused_normal_sums(px, pn, voxel, origin)
        assert np.array_equal(on[:, 0].cpu().numpy(), keys) and np.array_equal(on[:, 6:9].cpu().numpy(), sums)


def _inputs(case, seed=0):
    xyz, votes, thr, voxel = CLOUDS[case]
    n = len(xyz)
    rgb = np.random.default_rng(n).integers(0, 256, (n, 3)).astype(np.uint8)
    box = _box(xyz.min(0) - 0.013, xyz.max(0) + 0.021)
    return (_cuda(xyz), _cuda(rgb), _cuda(votes), _cuda(_unit_normals(n, seed))), thr, (lambda sess: sess.begin([box], voxel))


def _on_off(d, bounds, thr, begin, max_cells, mode=0, dedup=None):
    n_max = max(b - a for a, b in bounds)
    n_dedup = 0 if dedup is None else dedup.shape[0]
    on = NormalRanks(len(bounds), n_max, True, max_cells=max_cells, n_dedup=n_dedup)
    off = NormalRanks(len(bounds), n_max, False, max_cells=max_cells, n_dedup=n_dedup)
    parts = _parts(d, bounds)
    res_on = on.step(parts, thr, begin, mode=mode, dedup=dedup)
    res_off = off.step(parts, thr, begin, mode=mode, dedup=dedup)
    _same(res_on[0][:4], res_off[0])  # keys, xyz, rgb, count
    assert res_on[1] == res_off[1] and res_on[2] == res_off[2]  # counts after the partial and after the merge
    return on, res_on, res_off, parts


@pytest.mark.parametrize("R", [2, 3, 8, 16])
@pytest.mark.parametrize("form", ["dense", "hashed"])
def test_ranks_equal_one_gpu(lib_built, R, form):
    """Dense: a grid the sessions hold (ddn_fuse_merge_peers_normals).  Hashed: a grid beyond the sessions' bitmap (both
    forms enqueued, the hashed merge runs).  Uneven shares.  The concatenation equals the one-GPU normals result (dense and
    hashed) and the numpy statement; the records hold what they should."""
    case = "threshold_drops"
    d, thr, begin = _inputs(case, seed=R)
    bounds = _deal(d[0].shape[0], R)
    max_cells = 1 << 34 if form == "dense" else 1 << 20
    vr, (cat, part_counts, counts, recs), off, parts = _on_off(d, bounds, thr, begin, max_cells)
    assert all(s.grid_state().status == (0 if form == "dense" else 4) for s in vr.sessions)
    hashed, dense, grid = _one_gpu(*d, thr, begin)
    _same(cat, hashed)
    _same(cat, dense)
    _assert_oracle(cat, d[0], d[2], d[3], thr, grid)
    _assert_records(vr, recs, off[3], parts, thr, grid)


@pytest.mark.parametrize("skew", ["one_empty_one_full", "empty_ranks", "one_rank"])
@pytest.mark.parametrize("form", ["dense", "hashed"])
def test_skewed_shares(lib_built, skew, form):
    d, thr, begin = _inputs("many_voxels", seed=1)
    n = d[0].shape[0]
    R, frac = {"one_empty_one_full": (4, [0.0, 0.97, 0.02, 0.01]), "empty_ranks": (8, [0.3, 0.3, 0.4, 0, 0, 0, 0, 0]),
               "one_rank": (1, [1.0])}[skew]
    _, (cat, *_), _, _ = _on_off(d, _deal(n, R, frac), thr, begin, 1 << 34 if form == "dense" else 1 << 20)
    hashed, dense, grid = _one_gpu(*d, thr, begin)
    _same(cat, hashed)
    _same(cat, dense)


@pytest.mark.parametrize("form", ["dense", "hashed"])
def test_one_voxel_on_every_rank(lib_built, form):
    """Every rank holds a share of the same voxels, and one voxel with 800 points, split over all 8 ranks."""
    R, voxel = 8, 0.01
    rng = np.random.default_rng(3)
    line = (np.arange(60000, dtype=np.float32)[:, None] * np.float32(voxel) + 0.005) * np.array([[1, 0, 0]], np.float32)
    xyz = np.concatenate([np.tile(line, (R, 1)), np.full((R * 100, 3), 0.3051, np.float32)])
    xyz = xyz[rng.permutation(len(xyz))]
    rgb = rng.integers(0, 256, (len(xyz), 3)).astype(np.uint8)
    d = (_cuda(xyz), _cuda(rgb), _cuda(np.zeros(len(xyz), np.uint8)), _cuda(_unit_normals(len(xyz), 5)))
    box = _box(xyz.min(0) - 0.01, xyz.max(0) + 0.01)
    begin = lambda sess: sess.begin([box], voxel)
    _, (cat, *_), _, _ = _on_off(d, _deal(len(xyz), R, [1 / R] * R), 1, begin, 1 << 34 if form == "dense" else 1 << 16)
    hashed, dense, grid = _one_gpu(*d, 1, begin)
    _same(cat, hashed)
    _same(cat, dense)
    _assert_oracle(cat, d[0], d[2], d[3], 1, grid)
    assert int(cat[3].max()) >= R * 100


@pytest.mark.parametrize("R", [3, 8])
@pytest.mark.parametrize("mode", [0, 1])
def test_dedup_n5(lib_built, R, mode):
    """N5 at the owner (dense merge, mode 0) and through the tombstones of every rank (hashed, mode 1)."""
    d, thr, begin = _inputs("threshold_drops", seed=7)
    dedup = d[0][::37].contiguous()
    bounds = _deal(d[0].shape[0], R)
    _, (cat, *_), _, _ = _on_off(d, bounds, thr, begin, 1 << 34, mode=mode, dedup=dedup)
    hashed, dense, grid = _one_gpu(*d, thr, begin, dedup=dedup)
    _same(cat, hashed)
    _same(cat, dense)
    _assert_oracle(cat, d[0], d[2], d[3], thr, grid, dedup=dedup)


def test_support_vote_bytes(lib_built):
    """The consistency kernel's vote bytes of a min_support step (tested with the support-mode fusion threshold), dealt
    to the ranks by views: the one-GPU engine's voxels and normals."""
    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    res = _engine(voxel=0.02, min_support=2, support_tau=0.01, fuse_normals=True).run(*_scene_args(sc, nbr))
    thr = res.fusion_threshold()
    d = (res.xyz.view(-1, 3), res.grid_rgb().reshape(-1, 3).contiguous(), res.votes.view(-1), res.normals.view(-1, 3))
    per_view = res.xyz.shape[1] * res.xyz.shape[2]
    from depthdensifier_b200.distributed import shard_bounds

    views = [(a * per_view, b * per_view) for a, b in shard_bounds(res.xyz.shape[0], 3)]
    begin = lambda sess: sess.begin([res.bbox_valid], 0.02)
    _, (cat, *_), _, _ = _on_off(d, views, thr, begin, 1 << 34)
    _same(cat, (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.voxel_normal))


def test_dense_hashed_hashed_dense_steps(lib_built):
    """dense, hashed, hashed, dense on the same virtual ranks: every step equals the one-GPU engine's voxels and normals."""
    from depthdensifier_b200 import _lib
    from depthdensifier_b200.distributed import shard_bounds

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    args = _scene_args(sc, nbr)
    R, vr = 3, None
    for voxel, status in [(0.05, _lib.GRID_OK), (0.02, _lib.GRID_HASHED), (0.015, _lib.GRID_HASHED), (0.05, _lib.GRID_OK)]:
        res = _engine(max_cells=1 << 26, voxel=voxel, fuse_normals=True).run(*args)
        assert res.session.grid_state().status == status
        d = (res.xyz.view(-1, 3), res.grid_rgb().reshape(-1, 3).contiguous(), res.votes.view(-1), res.normals.view(-1, 3))
        per_view = res.xyz.shape[1] * res.xyz.shape[2]
        views = [(a * per_view, b * per_view) for a, b in shard_bounds(res.xyz.shape[0], R)]
        if vr is None:
            vr = NormalRanks(R, max(b - a for a, b in views), True, max_cells=1 << 26)

        def begin(sess, box=res.bbox_valid, voxel=voxel):
            sess.begin([box], voxel)

        cat, *_ = vr.step(_parts(d, views), res.vote_threshold, begin)
        assert all(s.grid_state().status == status for s in vr.sessions)
        _same(cat, (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.voxel_normal))
    for hf in vr.hfs:
        assert bool((hf.table == 255).all()) and bool((hf.slots[: hf.cap_voxels * 4] == 255).all())


@pytest.mark.parametrize("mode", [0, 1])
def test_flag_when_only_the_sum_reaches_2_24(lib_built, mode):
    """A voxel with fewer than 2^24 points on each of two ranks but 2^24 or more in all: the owner sets counts[0] = -1,
    on the dense merge (mode 0) and on the hashed one (mode 1)."""
    n = (1 << 23) + 4096
    xyz = np.full((2 * n, 3), 0.5, np.float32)
    xyz[-8:] = 3.0
    nrm = torch.zeros((2 * n, 3), dtype=torch.float32, device="cuda")
    nrm[:, 2] = 1.0
    d = (_cuda(xyz), torch.zeros((2 * n, 3), dtype=torch.uint8, device="cuda"), torch.zeros(2 * n, dtype=torch.uint8, device="cuda"), nrm)
    box = _box(np.zeros(3, np.float32), np.full(3, 4.0, np.float32))
    vr = NormalRanks(2, n, True, max_cells=1 << 20)
    cat, part_counts, counts, _ = vr.step(_parts(d, [(0, n), (n, 2 * n)]), 1, lambda s: s.begin([box], 1.0), mode=mode)
    assert all(p[0] == n for p in part_counts)
    assert int(cat[3][0]) == 2 * n - 8 and int(cat[3][1]) == 8
    assert sorted(c[0] for c in counts) == [-1, n]
    assert torch.equal(cat[4], torch.tensor([[0, 0, 1], [0, 0, 1]], dtype=torch.float32, device="cuda"))


def _sharded_inputs(sc):
    return tuple(t.cuda().contiguous() for t in (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets))


@pytest.mark.parametrize("scene", ["standard", "dome"])
@pytest.mark.parametrize("dedup", [False, True])
def test_sharded_one_rank_equals_engine(lib_built, scene, dedup):
    """ShardedDensifier with world 1 and fuse_normals: DensifyEngine's per-point normals, voxels and voxel normals, through
    run and through run_host (out["normal"])."""
    from depthdensifier_b200 import _lib, ops
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig

    kw = DOME if scene == "dome" else dict(n_views=6, width=203, height=131, n_sparse=700, seed=9)
    voxel = DOME_VOXEL if scene == "dome" else 0.02
    sc = make_scene(SceneConfig(**kw))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    V, H, W = sc.mono_depth.shape
    ref = _engine(voxel=voxel, dedup_sparse=dedup, fuse_normals=True).run(*_scene_args(sc, nbr))
    assert ref.session.grid_state().status == (_lib.GRID_HASHED if scene == "dome" else _lib.GRID_OK)
    cfg = DensifyConfig(voxel=voxel, dedup_sparse=dedup, fuse_normals=True,
                        align=ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True))
    sd = ShardedDensifier(cfg, "cuda", 0, 1, V, 0, V, sc.cam_from_world, sc.intrinsics, nbr, H, W)
    res = sd.run(*_sharded_inputs(sc))
    mv = res.check()
    assert mv == ref.voxel_keys.shape[0] and int(res.counts[0]) == int(ref.counts[0])
    assert torch.equal(res.normals, ref.normals)
    _same([t[:mv] for t in (res.voxel_keys, res.voxel_xyz, res.voxel_rgb, res.voxel_count, res.voxel_normal)],
          (ref.voxel_keys, ref.voxel_xyz, ref.voxel_rgb, ref.voxel_count, ref.voxel_normal))
    host = sd.pin_host_inputs(*(t.contiguous() for t in (sc.mono_depth, sc.normal, sc.mask, sc.rgb, sc.sparse_xyz, sc.sparse_offsets)))
    for _ in range(2):
        out = sd.run_host(*host, chunk_views=4)
        assert out["num_points"] == int(ref.counts[0])
        for name, t in (("keys", ref.voxel_keys), ("xyz", ref.voxel_xyz), ("rgb", ref.voxel_rgb), ("count", ref.voxel_count),
                        ("normal", ref.voxel_normal)):
            assert np.array_equal(out[name].numpy(), t.cpu().numpy()), name


def test_sharded_normals_without_fusion(lib_built):
    """fuse_normals without a voxel size: per-point normals only, as on one GPU."""
    from depthdensifier_b200 import ops
    from depthdensifier_b200.distributed import ShardedDensifier
    from depthdensifier_b200.engine import DensifyConfig

    sc = make_scene(SceneConfig(n_views=6, width=203, height=131, n_sparse=700, seed=9))
    nbr = nearest_views_table(sc.cam_from_world.numpy(), 4)
    V, H, W = sc.mono_depth.shape
    ref = _engine(voxel=None, fuse_normals=True).run(*_scene_args(sc, nbr))
    cfg = DensifyConfig(voxel=None, fuse_normals=True, align=ops.AlignOptions(adaptive_correspondences=False, zero_unmasked_passthrough=True))
    res = ShardedDensifier(cfg, "cuda", 0, 1, V, 0, V, sc.cam_from_world, sc.intrinsics, nbr, H, W).run(*_sharded_inputs(sc))
    assert torch.equal(res.normals, ref.normals) and res.voxel_normal is None and res.voxel_keys is None


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_ranks_equal_one_rank_with_normals(lib_built):
    """scripts/check_multi_gpu.py --fuse-normals under torchrun: the peer path, dense, dedup and hashed cases."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(ROOT / "scripts" / "check_multi_gpu.py"), "--fuse-normals"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=str(ROOT))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
    rep = json.loads(line)["multi_gpu_check"]
    assert all(r["passed"] for r in rep) and all(r["path"] == "peer" for r in rep), rep
    assert sum(1 for r in rep if r.get("fuse_normals")) == 3
