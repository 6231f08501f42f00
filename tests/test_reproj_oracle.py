"""The host restatement of the forward-backward reprojection check (tests/reproj_oracle.py): a rig whose supporting
entries are known in closed form, the explicit round trip against the closed form the kernel evaluates, and the
table rules it shares with the support count."""

import numpy as np
import pytest

import reproj_oracle as RO
import support_oracle as S
from test_support_oracle import BASE, F, H, W, Z0, plane_scene

# The translated-plane rig of test_support_oracle: view t, translated by b along x with depth Z0 (1 + delta), sends the
# round trip back f b |delta| / (Z0 (1 + delta)) pixels from where it started.
ERR1 = F * BASE * 0.005 / (Z0 * 1.005)  # view 1: 0.0274 px
ERR2 = F * BASE * 0.02 / (Z0 * 1.02)  # view 2: 0.1078 px


def _rig():
    refined, poses, intr, pts, px = plane_scene()
    return refined, poses, intr, pts, px, np.zeros(len(pts), dtype=np.int64)


@pytest.mark.parametrize("sample_mode", ["nearest", "bilinear"])
def test_reproj_counts_in_closed_form(sample_mode):
    refined, poses, intr, pts, px, src = _rig()
    in1 = (px >= 6).astype(np.int64)  # view 1 sees u = x - 5.5
    in2 = (px <= W - 6).astype(np.int64)  # view 2 sees u = x + 5.5
    _, py = RO.source_pixels(pts, poses[0], intr[0])
    nbr = np.array([[1, 2], [0, 2], [0, 1]], np.int32)
    kw = dict(support_tau=0.03, sample_mode=sample_mode)  # both neighbours pass the depth test
    for rho, want in ((0.5 * ERR1, 0 * in1), (0.5 * (ERR1 + ERR2), in1), (2 * ERR2, in1 + in2), (1.0, in1 + in2)):
        got, ties, frac, decided = RO.reproj_support_with_ties(pts, src, refined, poses, intr, nbr, reproj_px=rho, **kw)
        np.testing.assert_array_equal(got, want, err_msg=f"rho = {rho}")
        # the only ties: row 0, where v = 0 lies on the border band; the pairs the pixel bound decides are the rest
        assert frac == pytest.approx(1 / H) and np.array_equal(ties > 0, py == 0)
        assert decided == int(((in1 + in2 - want) * (py > 0)).sum())
    # the depth test still applies: at tau = 0.01 view 2 (2 % off) never supports, whatever rho
    got = RO.consistency_support_reproj(pts, src, refined, poses, intr, nbr, support_tau=0.01, reproj_px=1e30,
                                        sample_mode=sample_mode)
    np.testing.assert_array_equal(got, in1)


@pytest.mark.parametrize("sample_mode", ["nearest", "bilinear"])
@pytest.mark.parametrize("tau", [0.004, 0.01, 0.03])
def test_huge_rho_is_the_support_count(sample_mode, tau):
    refined, poses, intr, pts, px, src = _rig()
    nbr = np.array([[1, 2], [0, 2], [0, 1]], np.int32)
    want = S.consistency_support(pts, src, refined, poses, intr, nbr, support_tau=tau, sample_mode=sample_mode)
    got = RO.consistency_support_reproj(pts, src, refined, poses, intr, nbr, support_tau=tau, reproj_px=1e30,
                                        sample_mode=sample_mode)
    np.testing.assert_array_equal(got, want)


def test_own_view_padding_and_repeats():
    """Own-view entries and -1 padding never count; a view listed twice counts twice."""
    refined, poses, intr, pts, px, src = _rig()
    in1 = (px >= 6).astype(np.int64)
    kw = dict(support_tau=0.03, reproj_px=0.5 * (ERR1 + ERR2))
    nbr = np.array([[0, 1, -1, 1, 2], [0, 2, -1, -1, -1], [0, 1, -1, -1, -1]], np.int32)
    np.testing.assert_array_equal(RO.consistency_support_reproj(pts, src, refined, poses, intr, nbr, **kw), 2 * in1)
    nbr = np.array([[0, -1], [0, 2], [0, 1]], np.int32)
    np.testing.assert_array_equal(RO.consistency_support_reproj(pts, src, refined, poses, intr, nbr, **kw), 0 * in1)


def _random_camera(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    a, b, c, d = q
    Rm = np.array([[a * a + b * b - c * c - d * d, 2 * (b * c - a * d), 2 * (b * d + a * c)],
                   [2 * (b * c + a * d), a * a - b * b + c * c - d * d, 2 * (c * d - a * b)],
                   [2 * (b * d - a * c), 2 * (c * d + a * b), a * a - b * b - c * c + d * d]])
    pose = np.concatenate([Rm, rng.normal(size=(3, 1)) * 2], axis=1)
    intr = np.array([rng.uniform(200, 2000), rng.uniform(200, 2000), rng.uniform(100, 1000), rng.uniform(100, 800)])
    return pose, intr


def test_explicit_round_trip_is_the_closed_form():
    """On random pose pairs, intrinsics, pixels and depths, the explicit float64 round trip equals the closed form of
    include/ddn_b200.h: z' = d + w (e_z - d), (x' - x, y' - y) = w (d e_x - P e_z, d e_y - Q e_z) / (d z')."""
    rng = np.random.default_rng(7)
    worst = 0.0
    for _ in range(2000):
        (ps, ks), (pt, kt) = _random_camera(rng), _random_camera(rng)
        x, y, d = rng.uniform(0, 2000), rng.uniform(0, 1500), rng.uniform(0.5, 50)
        P, Q = d * x, d * y
        Kinv = np.linalg.inv(RO.R.kmatrix(ks))
        X = ps[:, :3].T @ (Kinv @ np.array([P, Q, d]) - ps[:, 3])  # world point of pixel (x, y) at depth d
        u, v, z = RO.project(X[None], pt, kt)
        D = z[0] * rng.uniform(0.8, 1.2)
        xp, yp, zp = (a[0] for a in RO.forward_backward(u, v, np.array([D]), pt, kt, ps, ks))
        z = z[0]
        e = RO.epipole_f64(ps, ks, pt)
        w = (z - D) / z
        zc = d + w * (e[2] - d)
        dx, dy = w * (d * e[0] - P * e[2]) / (d * zc), w * (d * e[1] - Q * e[2]) / (d * zc)
        for a, b in ((zp, zc), (xp - x, dx), (yp - y, dy)):
            worst = max(worst, abs(a - b) / max(abs(a), abs(b), 1e-300))
    assert worst < 1e-9, worst


def test_host_epipole_replay_is_float32_accurate():
    """The replay of K4's float32 epipole from the host tables lands within float32 accuracy of the exact epipole."""
    rng = np.random.default_rng(3)
    cams = [_random_camera(rng) for _ in range(12)]
    poses, intr = np.stack([c[0] for c in cams]), np.stack([c[1] for c in cams])
    src, c = RO.host_tables(poses, intr)
    for s in range(12):
        for t in range(12):
            if s != t:
                e = RO.epipole_f64(poses[s], intr[s], poses[t])
                de = RO.epipole_error(src[s], c[t], poses[s], intr[s], poses[t])
                assert (de <= 1e-5 * (np.abs(e).max() + intr[s].max())).all()
