"""The host restatement of the multi-view support count (tests/support_oracle.py) on a scene whose counts are known in
closed form, and the vote-byte encoding that carries the support keep rule to the fusion passes."""

import numpy as np
import pytest

from oracle import restatement as R
import support_oracle as S

W, H, F, Z0 = 64, 48, 100.0, 2.0
BASE = 0.11  # camera x offsets of views 1 and 2: the plane moves by F * BASE / Z0 = 5.5 px, so no point lands on a border


def plane_scene():
    """Three cameras looking down +z at the plane z = Z0, translated along x (0, +BASE, -BASE).  View 1's depth is the
    true depth times 1.005, view 2's times 1.02; view 0's is exact."""
    poses = np.zeros((3, 3, 4))
    for v, cx in enumerate((0.0, BASE, -BASE)):
        poses[v, :, :3] = np.eye(3)
        poses[v, 0, 3] = -cx
    intr = np.tile(np.array([F, F, W / 2, H / 2]), (3, 1))
    refined = np.stack([np.full((H, W), Z0 * s, np.float32) for s in (1.0, 1.005, 1.02)])
    pts, pyv, pxv = R.backproject_view(refined[0], intr[0], poses[0])
    return refined, poses, intr, pts, pxv


@pytest.mark.parametrize("sample_mode", ["nearest", "bilinear"])
def test_support_counts_in_closed_form(sample_mode):
    refined, poses, intr, pts, px = plane_scene()
    src = np.zeros(len(pts), dtype=np.int64)
    in1 = px >= 6  # view 1 sees u = x - 5.5
    in2 = px <= W - 6  # view 2 sees u = x + 5.5
    kw = dict(sample_mode=sample_mode)
    # eps = 0.01 splits the two neighbours: 0.5 % agrees, 2 % does not
    nbr = np.array([[1, 2], [0, 2], [0, 1]], np.int32)
    got = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=0.01, **kw)
    np.testing.assert_array_equal(got, in1.astype(np.int64))
    got = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=0.03, **kw)
    np.testing.assert_array_equal(got, in1.astype(np.int64) + in2)
    got = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=0.004, **kw)
    np.testing.assert_array_equal(got, np.zeros(len(pts), np.int64))
    # own-view entries and -1 padding never count; a repeated entry counts once per entry
    nbr = np.array([[0, 1, -1, 1], [0, 2, -1, -1], [0, 1, -1, -1]], np.int32)
    got = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=0.01, **kw)
    np.testing.assert_array_equal(got, 2 * in1.astype(np.int64))
    nbr = np.array([[0, -1], [0, 2], [0, 1]], np.int32)
    got = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=0.03, **kw)
    np.testing.assert_array_equal(got, np.zeros(len(pts), np.int64))


@pytest.mark.parametrize("sample_mode", ["nearest", "bilinear"])
def test_support_of_view_needs_a_depth(sample_mode):
    """A neighbour without depth where the point lands (D = 0; bilinear: any of the four taps 0) never supports it,
    whatever tau."""
    refined, poses, intr, pts, px = plane_scene()
    hole = refined[1].copy()
    hole[:, : W // 2] = 0
    ok = S.support_of_view(pts, hole, poses[1], intr[1], support_tau=10.0, sample_mode=sample_mode)
    u = px - 5.5
    np.testing.assert_array_equal(ok, u >= W // 2)


@pytest.mark.parametrize("thr", [0, 1, 5, 254, 255, 1000])
@pytest.mark.parametrize("m", [0, 1, 2, 40])
def test_vote_byte_encodes_the_keep_rule(thr, m):
    """byte < min(thr, 254) is the keep rule at every threshold and minimum support, and with m = 0 and thr <= 254 the
    byte is the plain vote byte min(votes, 254)."""
    rng = np.random.default_rng(thr * 7 + m)
    votes = rng.integers(0, 400, 5000)
    support = rng.integers(0, 60, 5000)
    byte = S.encode_votes(votes, support, thr, m)
    np.testing.assert_array_equal(byte < min(thr, 254), S.keep(votes, support, thr, m))
    assert (byte != 255).all()
    if m == 0 and thr <= 254:
        np.testing.assert_array_equal(byte, np.minimum(votes, 254))
