"""The forward-backward reprojection check of ddn_backproject_filter_support_reproj (parity unpinned: no reference
implementation), restated on the host.

Built on tests/support_oracle.py and oracle/restatement.py's per-view functions.  For a point of source view s at pixel
(x, y) and a neighbour entry t: (u, v, z) and D as ``support_oracle`` has them; then, EXPLICITLY in float64, the pixel
(u, v) of t (continuous coordinates, in both sampling modes) is back-projected at depth D, taken to the world and into
s, and projected: (x', y'), z'.  t supports the point iff the depth test of ``support_oracle`` holds, z' > 0 and
|(x', y') - (x, y)| <= rho.  The closed form the kernel evaluates (include/ddn_b200.h) is not used here, so that the
tests check its derivation."""

from __future__ import annotations

import numpy as np

from oracle import restatement as R
from parity import EPS_PX, EPS_REL, EPS_Z
import support_oracle as S


def project(world, pose, intr):
    """(u, v, z) of world points [N,3] in a view, with u = U / z exactly (restatement.project_points divides by
    z + 1e-8, the reference's quirk, which would bias a sub-pixel round trip)."""
    cam = world @ pose[:, :3].T + pose[:, 3]
    z = cam[:, 2]
    return intr[0] * cam[:, 0] / z + intr[2], intr[1] * cam[:, 1] / z + intr[3], z


def forward_backward(u, v, D, pose_t, intr_t, pose_s, intr_s):
    """(x', y', z'): t's pixel (u, v) at depth D, back-projected, taken to the world and projected into s (float64).
    pose_s [3,4] and intr_s [4], or one per point ([N,3,4], [N,4])."""
    fx, fy, cx, cy = (float(a) for a in intr_t)
    cam_t = np.stack([(u - cx) / fx * D, (v - cy) / fy * D, D], axis=1)
    Rt, tt = pose_t[:, :3], pose_t[:, 3]
    world = (cam_t - tt) @ Rt  # R_t^T (X - t_t), row-wise
    if pose_s.ndim == 2:
        return project(world, pose_s, intr_s)
    cam = np.einsum("nij,nj->ni", pose_s[:, :, :3], world) + pose_s[:, :, 3]
    z = cam[:, 2]
    return intr_s[:, 0] * cam[:, 0] / z + intr_s[:, 2], intr_s[:, 1] * cam[:, 1] / z + intr_s[:, 3], z


def source_pixels(points, pose_s, intr_s):
    """The integer pixel (x, y) each point was back-projected from (projected back into its view and rounded)."""
    x, y, _ = project(points, pose_s, intr_s)
    return np.rint(x), np.rint(y)


# ---- the float32 error of the epipole K4 uses (filter.cu: epipole) ----

def host_tables(poses, intr):
    """The float32 table values the epipole reads, computed as build_pair_tables does: src [V,16] (rows of
    R_s^T K_s^-1 with c_s, then cx, cy, fx, fy) and c [V,3] (camera centres, floats 12-14 of a pair-table entry)."""
    V = len(poses)
    src = np.zeros((V, 16), np.float32)
    c = np.zeros((V, 3), np.float32)
    for s in range(V):
        Rs, ts = poses[s][:, :3], poses[s][:, 3]
        fx, fy, cx, cy = (float(a) for a in intr[s])
        for i in range(3):
            r0, r1, r2 = Rs[0, i], Rs[1, i], Rs[2, i]
            src[s, i * 4:i * 4 + 4] = [r0 / fx, r1 / fy, -r0 * cx / fx - r1 * cy / fy + r2, -(r0 * ts[0] + r1 * ts[1] + r2 * ts[2])]
        src[s, 12:16] = [cx, cy, fx, fy]
        c[s] = -(Rs.T @ ts)
    return src, c


def device_tables(pair_table, src_table):
    """(src [n_src,16], {(s, t): c_t}) from the downloaded tables of ddn_build_pair_tables* (the hot entries of each
    row: floats 12-14 carry c_t, float 15 t, entry 0's float 22 the hot count)."""
    pt = np.asarray(pair_table, np.float32)
    n_src = pt.shape[0]
    ct = {}
    for s in range(n_src):
        n_hot = int(pt[s, 0, 22:23].view(np.int32)[0])
        for k in range(n_hot):
            t = int(pt[s, k, 15:16].view(np.int32)[0])
            ct[(s, t)] = pt[s, k, 12:15].copy()
    return np.asarray(src_table, np.float32), ct


def epipole_f32(src, ct):
    """K4's float32 epipole of t in s, replayed operation for operation (each rounded, no contraction)."""
    f = np.float32
    fx, fy, cx, cy = src[14], src[15], src[12], src[13]
    a0 = a1 = a2 = f(0)
    for i in range(3):
        m0, m1, m2 = src[i * 4], src[i * 4 + 1], src[i * 4 + 2]
        ra, rb = f(m0 * fx), f(m1 * fy)
        rc = f(f(m2 + f(m0 * cx)) + f(m1 * cy))
        c = f(ct[i] - src[i * 4 + 3])
        a0, a1, a2 = f(a0 + f(ra * c)), f(a1 + f(rb * c)), f(a2 + f(rc * c))
    return np.array([f(f(fx * a0) + f(cx * a2)), f(f(fy * a1) + f(cy * a2)), a2], np.float64)


def epipole_f64(pose_s, intr_s, pose_t):
    """e = K_s (R_s c_t + t_s) in float64."""
    c_t = -pose_t[:, :3].T @ pose_t[:, 3]
    return R.kmatrix(intr_s) @ (pose_s[:, :3] @ c_t + pose_s[:, 3])


def epipole_error(src_row, ct, pose_s, intr_s, pose_t):
    """|e32 - e64| per component: the kernel's epipole against the exact one."""
    return np.abs(epipole_f32(src_row, ct) - epipole_f64(pose_s, intr_s, pose_t))


# ---- per (point, entry) decisions with tie bands ----

def pair_reproj_ties(points, xs, ys, pose_s, intr_s, refined_t, pose_t, intr_t, e, de, support_tau=0.01, reproj_px=1.0,
                     sample_mode="nearest"):
    """(support[N], tie[N], decided[N]) of all points (pixels xs, ys of their source views s) against neighbour view t.
    pose_s [N,3,4], intr_s [N,4]: each point's source view; e, de [N,3]: t's epipole in it (float64) and the error of
    K4's float32 epipole |e32 - e64|.  decided: the depth test passes and the reprojection test fails, both outside
    their tie bands.

    Tie bands: those of ``support_oracle.pair_support_ties``, plus a band around |(x', y') - (x, y)| = rho derived from
    the device's errors.  Writing err = |w| |(e_x - x e_z, e_y - y e_z)| / |z'| with w = (z - D)/z (the closed form):
      * z and D: the depth band on z - D (EPS_REL * D; bilinear: plus the sub-pixel error times the tap slope), carried
        through d err / d(z - D) = err / |z - D|;
      * the float32 epipole: |w| |(de_x + |x| de_z, de_y + |y| de_z)| / |z'| + err |w| de_z / |z'|;
      * the float32 rounding of the closed form: 2^-23 relative on each of A, B (|w| |(|e_x| + |x e_z|, |e_y| + |y e_z|)|
        2^-23 / |z'|) and 2^-20 relative on err for the dozen roundings of the rest."""
    h, w = refined_t.shape
    n = len(points)
    _, det = R.votes_against_view(points, np.zeros((n, 3)), refined_t, pose_t, intr_t, grazing=-np.inf,
                                  sample_mode=sample_mode, return_detail=True)
    u, v, z, inb = det["u"], det["v"], det["z"], det["inb"]
    ue, ve, _ = project(points, pose_t, intr_t)  # the continuous (u, v) of the round trip, without the 1e-8 quirk
    tau32 = np.float32(support_tau)
    e, de = e.T, de.T
    tie = (np.abs(u) < EPS_PX) | (np.abs(u - w) < EPS_PX) | (np.abs(v) < EPS_PX) | (np.abs(v - h) < EPS_PX)
    tie |= np.abs(z) < EPS_Z

    def decide(x0, y0):
        ok = inb & (x0 >= 0) & (x0 < w) & (y0 >= 0) & (y0 < h)
        if sample_mode == "nearest":
            D32 = np.zeros(n, np.float32)
            D32[ok] = refined_t[y0[ok], x0[ok]]
            valid = ok & (D32 > 0)
            D = D32.astype(np.float64)
            q = np.abs(z - D) - (tau32 * D32).astype(np.float64)
            band = EPS_REL * D
        else:
            x0c, y0c = np.clip(x0, 0, w - 1), np.clip(y0, 0, h - 1)
            x1c, y1c = np.clip(x0 + 1, 0, w - 1), np.clip(y0 + 1, 0, h - 1)
            taps = np.stack([refined_t[y0c, x0c], refined_t[y0c, x1c], refined_t[y1c, x0c], refined_t[y1c, x1c]]).astype(np.float64)
            fx, fy = u - x0, v - y0
            D = (1 - fx) * (1 - fy) * taps[0] + fx * (1 - fy) * taps[1] + (1 - fx) * fy * taps[2] + fx * fy * taps[3]
            valid = ok & (taps > 0).all(0)
            q = np.abs(z - D) - tau32 * D
            band = EPS_REL * np.abs(D) + EPS_PX * 2 * (taps.max(0) - taps.min(0))
        with np.errstate(all="ignore"):
            xp, yp, zp = forward_backward(ue, ve, D, pose_t, intr_t, pose_s, intr_s)
            err = np.hypot(xp - xs, yp - ys)
            om = np.abs((z - D) / z)
            b = np.where(z != D, err * band / np.abs(z - D), 0.0)
            b += om * np.hypot(de[0] + np.abs(xs) * de[2], de[1] + np.abs(ys) * de[2]) / np.abs(zp) + err * om * de[2] / np.abs(zp)
            b += om * np.hypot(np.abs(e[0]) + np.abs(xs * e[2]), np.abs(e[1]) + np.abs(ys * e[2])) * 2.0 ** -23 / np.abs(zp)
            b += err * 2.0 ** -20
            r_ok = (zp > 0) & (err <= reproj_px)
            r_near = (zp > 0) & (np.abs(err - reproj_px) < b)
        d_ok, d_near = valid & (q <= 0), valid & (np.abs(q) < band)
        sup = d_ok & r_ok
        near = (d_near & (r_ok | r_near)) | (r_near & (d_ok | d_near))
        return sup, near, d_ok & ~d_near & ~r_ok & ~r_near

    x0 = np.floor(np.where(inb, u, 0)).astype(int)
    y0 = np.floor(np.where(inb, v, 0)).astype(int)
    base, near, decided = decide(x0, y0)
    tie |= near
    fu, fv = u - np.floor(u), v - np.floor(v)
    for du, dv, sel in (
        (-1, 0, fu < EPS_PX), (1, 0, fu > 1 - EPS_PX), (0, -1, fv < EPS_PX), (0, 1, fv > 1 - EPS_PX),
        (-1, -1, (fu < EPS_PX) & (fv < EPS_PX)), (1, 1, (fu > 1 - EPS_PX) & (fv > 1 - EPS_PX)),
        (-1, 1, (fu < EPS_PX) & (fv > 1 - EPS_PX)), (1, -1, (fu > 1 - EPS_PX) & (fv < EPS_PX)),
    ):
        sel = sel & inb
        if sel.any():
            alt, near_alt, _ = decide(x0 + du, y0 + dv)
            tie |= sel & ((alt != base) | near_alt)
    return base, tie, decided & ~tie


def reproj_support_with_ties(points, src_view, refined_all, poses, intr, nbr, support_tau=0.01, reproj_px=1.0,
                             sample_mode="nearest", tables=None):
    """(support[N] int64, ties[N] int64, pair tie fraction, decided): supporting entries of every point under the
    combined test (not saturated), entries per point inside a tie band, their share of the tested (point, entry) pairs,
    and the number of tie-free pairs the pixel bound decides (depth test passes, reprojection test fails).
    ``tables``: None (the epipole error from host-built float32 tables) or the downloaded (pair_table, src_table) of
    the call, rows indexed by source view.  ``refined_all``: [V,H,W] or a list of V maps of their own sizes."""
    V = len(refined_all)
    mult = S.table_multiplicity(nbr, V)
    if tables is None:
        src32, c32 = host_tables(poses, intr)
        ct = lambda s, t: c32[t]
    else:
        src32, cmap = device_tables(*tables)
        ct = lambda s, t: cmap[(s, t)]
    n = len(points)
    xs, ys = np.zeros(n), np.zeros(n)
    for s in np.unique(src_view):
        on_s = src_view == s
        xs[on_s], ys[on_s] = source_pixels(points[on_s], poses[s], intr[s])
    support = np.zeros(n, dtype=np.int64)
    ties = np.zeros(n, dtype=np.int64)
    pairs = decided = 0
    for t in range(V):
        sel = np.where(mult[src_view, t] > 0)[0]
        if len(sel) == 0:
            continue
        sv = src_view[sel]
        e_s, de_s = {}, {}
        for s in np.unique(sv):
            e_s[s] = epipole_f64(poses[s], intr[s], poses[t])
            de_s[s] = epipole_error(src32[s], ct(s, t), poses[s], intr[s], poses[t])
        e = np.stack([e_s[s] for s in sv])
        de = np.stack([de_s[s] for s in sv])
        ok, tie, dec = pair_reproj_ties(points[sel], xs[sel], ys[sel], np.asarray(poses)[sv], np.asarray(intr)[sv],
                                        refined_all[t], poses[t], intr[t], e, de, support_tau, reproj_px, sample_mode)
        m = mult[sv, t]
        support[sel] += ok * m
        ties[sel] += tie * m
        pairs += int(m.sum())
        decided += int((dec * m).sum())
    return support, ties, float(ties.sum()) / max(pairs, 1), decided


def consistency_support_reproj(points, src_view, refined_all, poses, intr, nbr, support_tau=0.01, reproj_px=1.0,
                               sample_mode="nearest"):
    """The support count under the combined test (``consistency_support`` with the reprojection check)."""
    return reproj_support_with_ties(points, src_view, refined_all, poses, intr, nbr, support_tau, reproj_px, sample_mode)[0]
