"""Host-side checks of the hashed multi-GPU fusion: sizing and argument checks of its entry points, and the numpy
statement of how the owners split the key space (tests/hashed_plan.py) on hand-built record sets."""

import ctypes

import numpy as np
import pytest

from hashed_plan import cut, samples_of, share_bound, shares, splitters

U64_MAX = np.uint64(2**64 - 1)


def test_merge_scratch_sizes_and_capacity(lib_built):
    from depthdensifier_b200 import _lib, ops

    lib = _lib.load()
    out = ctypes.c_int64(0)
    for R, cap in [(1, 1), (2, 1000), (8, 123457), (16, 1 << 30)]:
        assert lib.ddn_fuse_merge_hashed_scratch_bytes(R, cap, ctypes.byref(out)) == 0
        assert out.value >= cap * 48 + R * (_lib.HASH_SAMPLES + 1) * 8 + 17 * 8 + 32 * 8
    for R, cap in [(0, 10), (17, 10), (2, 0), (2, 1 << 31)]:
        assert lib.ddn_fuse_merge_hashed_scratch_bytes(R, cap, ctypes.byref(out)) == -1
    assert lib.ddn_fuse_merge_hashed_scratch_bytes(2, 10, None) == -1
    assert ops.hashed_merge_capacity(1000, 8) == 1000 + 4 + 16
    assert ops.hashed_merge_capacity(10**7, 8) == 10**7 + -(-16 * 10**7 // 4096) + 16


def test_entry_points_reject_bad_arguments(lib_built):
    """Invalid calls fail before any launch (no device needed)."""
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    sess, hf = _lib.FuseSession(), _lib.HashFuse()
    assert lib.ddn_fuse_finish_hashed_partial(ctypes.byref(sess), ctypes.byref(hf), 0, 10, 0, None, None, None, 1, None, 0, None, 10, None,
                                              None, 0, None) == -1
    assert b"invalid argument" in lib.ddn_last_error_string()
    ptrs = (ctypes.c_void_p * 2)(16, 32)
    assert lib.ddn_fuse_merge_hashed_peers(ctypes.byref(sess), ctypes.byref(hf), 0, 2, ptrs, ptrs, None, None, 0, None, None, None, None, 10,
                                           None) == -1
    # plausible buffers (never dereferenced: every check runs on the host first)
    sizes = [ctypes.c_int64(0) for _ in range(5)]
    assert lib.ddn_hash_fuse_sizes(1000, *[ctypes.byref(x) for x in sizes]) == 0
    hf = _lib.HashFuse(4096, 8192, 12288, 16384, 20480, sizes[0].value, 1000)
    sess = _lib.FuseSession(256, 512, 2048, None, 768, 1024, 1280)
    base = dict(mode=0, n=10, row_len=0, xyz=16, rgb=32, votes=None, thr=1, dedup=None, n_dedup=0, records=4096, cap_records=10,
                samples=8192, accum=12288, accum_bytes=10 * 40 + 16)

    def partial(**kw):
        a = {**base, **kw}
        return lib.ddn_fuse_finish_hashed_partial(ctypes.byref(sess), ctypes.byref(hf), a["mode"], a["n"], a["row_len"], a["xyz"], a["rgb"],
                                                  a["votes"], a["thr"], a["dedup"], a["n_dedup"], a["records"], a["cap_records"],
                                                  a["samples"], a["accum"], a["accum_bytes"], None)

    for bad, msg in [(dict(mode=2), b"mode"), (dict(n=-1), b"n_points"), (dict(n=990, n_dedup=20, dedup=16), b"cap_voxels"),
                     (dict(records=4100), b"16-byte"), (dict(samples=None), b"samples"), (dict(accum_bytes=100), b"accumulator"),
                     (dict(n_dedup=3), b"dedup"), (dict(cap_records=0), b"cap_records"), (dict(xyz=None), b"null")]:
        assert partial(**bad) == -1, bad
        assert msg in lib.ddn_last_error_string(), (bad, lib.ddn_last_error_string())

    def merge(rank=0, R=2, cap=100, scratch_bytes=1 << 30, plan=64, peers=ptrs):
        return lib.ddn_fuse_merge_hashed_peers(ctypes.byref(sess), ctypes.byref(hf), rank, R, peers, peers, plan, 16384, scratch_bytes, 16, 32,
                                               48, 64, cap, None)

    for bad, msg in [(dict(rank=2), b"rank"), (dict(R=17), b"rank"), (dict(cap=1001), b"cap_voxels"), (dict(cap=0), b"cap_out"),
                     (dict(scratch_bytes=1000), b"scratch"), (dict(plan=None), b"null"), (dict(peers=(ctypes.c_void_p * 2)(16, 0)), b"peer")]:
        assert merge(**bad) == -1, bad
        assert msg in lib.ddn_last_error_string(), (bad, lib.ddn_last_error_string())


def _keys(*vals):
    return np.unique(np.asarray(vals, dtype=np.uint64))


def _check(ranks, S):
    R = len(ranks)
    total = sum(len(k) for k in ranks)
    k = splitters(ranks, S)
    assert all(k[b] <= k[b + 1] for b in range(R))
    for q in ranks:  # the window search is the exact cut
        for key in k:
            assert cut(q, key, S) == int(np.searchsorted(q, key, side="left"))
    sh = shares(ranks, S)
    got = [sum(c for _, c in row) for row in sh]
    assert sum(got) == total
    for g in got:
        assert g <= share_bound(total, R, S)
    # every key goes to exactly one owner, the same for every rank that holds it
    owner = {}
    for b, row in enumerate(sh):
        for q, (begin, count) in enumerate(row):
            for key in ranks[q][begin:begin + count]:
                assert owner.setdefault(int(key), b) == b
    return got


@pytest.mark.parametrize("S", [4, 8, 4096])
def test_splitters_and_cuts(S):
    rng = np.random.default_rng(S)
    # uneven ranks, shared keys
    base = np.unique(rng.integers(0, 1 << 40, 5000).astype(np.uint64))
    ranks = [np.unique(rng.choice(base, n)) for n in (3000, 40, 1200, 2500)]
    _check(ranks, S)
    # empty ranks, and all empty
    _check([np.zeros(0, np.uint64), ranks[0], np.zeros(0, np.uint64), ranks[2]], S)
    assert _check([np.zeros(0, np.uint64)] * 3, S) == [0, 0, 0]
    # every rank holds the same keys (duplicates across ranks), and one key everywhere
    _check([base[:777]] * 5, S)
    _check([_keys(42)] * 8, S)
    # fewer records than samples, one rank only
    _check([_keys(5, 9), _keys(1, 2, 3)], S)
    _check([base], S)


def test_adversarial_rank_between_two_samples():
    """All of rank 1's records between two consecutive samples of rank 0: the bound still holds."""
    S = 16
    r0 = np.arange(0, 64 * 1000, 64, dtype=np.uint64)
    r1 = np.arange(64 * 500 + 1, 64 * 500 + 1 + 60, dtype=np.uint64)
    r1 = np.unique(np.concatenate([r1, r1 + np.uint64(64 * 62)]))  # two gaps of r0's samples, 120 keys
    s0 = samples_of(r0, S)
    assert np.searchsorted(s0, r1.min()) == np.searchsorted(s0, r1[59])  # the first 60 lie between two samples
    got = _check([r0, r1, r0[::7], np.zeros(0, np.uint64)], S)
    assert max(got) > 0
