"""Tie-aware comparison of CUDA consistency votes with the float64 oracle.

The reference evaluates stage 3 in float64 (scripts/test.py:58-76, 273-330); the CUDA kernel works in
float32 with float64-precomputed transforms.  The two can only disagree on a (point, view) pair whose
float64 quantities sit within a small band of a decision boundary.  The bands are STATED here:

  EPS_PX   pixel band around image borders and around integer pixel coordinates (truncation)
  EPS_DOT  band around the grazing threshold 0.087
  EPS_REL  relative band around z = depth_threshold * D
  EPS_Z    band around z = 0

A truncation-band pair only counts as a tie if one of the candidate pixels it could fall into
changes the decision.  Everything outside the bands must match bit for bit."""

from __future__ import annotations

import numpy as np

from oracle import restatement as R

EPS_PX = 4e-3
EPS_DOT = 2e-5
EPS_REL = 2e-5
EPS_Z = 1e-5


def pair_ties(points, normals, src_view, t, refined_t, pose_t, intr_t, depth_threshold=0.7, grazing=0.087,
              two_sided_tau=None):
    """Returns (vote[N] bool, tie[N] bool) of all points against target view t (nearest mode), one-sided
    (z < float32(thr * D)) or two-sided (|z - D| > float32(tau) * D); the threshold band is EPS_REL * D in both."""
    h, w = refined_t.shape
    vote, det = R.votes_against_view(points, normals, refined_t, pose_t, intr_t, depth_threshold=depth_threshold,
                                     grazing=grazing, two_sided_tau=two_sided_tau, return_detail=True)
    u, v, z, dot = det["u"], det["v"], det["z"], det["dot"]
    own = src_view == t
    tie = np.zeros(len(points), dtype=bool)
    near_border = (np.abs(u) < EPS_PX) | (np.abs(u - w) < EPS_PX) | (np.abs(v) < EPS_PX) | (np.abs(v - h) < EPS_PX)
    tie |= near_border & ~own
    tie |= np.abs(z) < EPS_Z
    tie |= np.abs(dot - grazing) < EPS_DOT
    # decision with the looked-up depth D
    thr32 = np.float32(depth_threshold)
    tau32 = None if two_sided_tau is None else np.float32(two_sided_tau)

    def test(D):
        """(decision, near-threshold flag) for looked-up depths D (float32; 0 where the lookup is invalid)."""
        D64 = D.astype(np.float64)
        if tau32 is None:
            return (D > 0) & (z < (thr32 * D)), (D > 0) & (np.abs(z - thr32 * D64) < EPS_REL * D64)
        q = np.abs(z - D64) - (tau32 * D).astype(np.float64)
        return (D > 0) & (q > 0), (D > 0) & (np.abs(q) < EPS_REL * D64)

    def decide(ui, vi):
        ok = (ui >= 0) & (ui < w) & (vi >= 0) & (vi < h)
        D = np.zeros(len(points), dtype=np.float32)
        D[ok] = refined_t[vi[ok], ui[ok]]
        dec, near_thr = test(D)
        return ok & dec, ok & near_thr

    cand = det["inb"] & ~own
    ui = np.where(cand, u, 0).astype(int)
    vi = np.where(cand, v, 0).astype(int)
    base, near = decide(ui, vi)
    tie |= cand & near
    fu = u - np.floor(u)
    fv = v - np.floor(v)
    for du, dv, sel in (
        (-1, 0, fu < EPS_PX), (1, 0, fu > 1 - EPS_PX), (0, -1, fv < EPS_PX), (0, 1, fv > 1 - EPS_PX),
        (-1, -1, (fu < EPS_PX) & (fv < EPS_PX)), (1, 1, (fu > 1 - EPS_PX) & (fv > 1 - EPS_PX)),
        (-1, 1, (fu < EPS_PX) & (fv > 1 - EPS_PX)), (1, -1, (fu > 1 - EPS_PX) & (fv < EPS_PX)),
    ):
        sel = sel & cand
        if sel.any():
            alt, near_alt = decide(ui + du, vi + dv)
            tie |= sel & ((alt != base) | near_alt)
    # own view: u = x*(1 - 1e-8/z) sits a deterministic ~1e-9 px below the integer x, so the lookup
    # pixel is (x-1, y-1) except in column/row 0 where float64 round-off decides (tie); otherwise
    # only the threshold band applies
    if own.any():
        tie |= own & det["inb"] & test(det["D"])[1]
        tie |= own & ((np.abs(u) < 0.5) | (np.abs(v) < 0.5))
    return vote, tie


def pair_ties_bilinear(points, normals, src_view, t, refined_t, pose_t, intr_t, depth_threshold=0.7, grazing=0.087,
                       two_sided_tau=None):
    """(vote[N] bool, tie[N] bool) against target view t for the bilinear sampling mode (N3), one- or two-sided.

    Bilinear D is continuous in (u, v) inside a cell, so the float32 kernel and the float64 statement can only
    disagree (i) in the border / z / grazing bands of the nearest mode, (ii) where (u, v) is within EPS_PX of an
    integer coordinate AND the neighbouring cell's tap set changes the outcome (the "all four taps > 0" rule is
    not continuous), (iii) where the compared quantity is within a band of its threshold.  That band has two
    terms: EPS_REL * D for the float32 products, and EPS_PX * 2 * (largest - smallest tap) for the sub-pixel
    error of (u, v) multiplied by the local depth slope (large across a depth discontinuity)."""
    h, w = refined_t.shape
    vote, det = R.votes_against_view(points, normals, refined_t, pose_t, intr_t, depth_threshold=depth_threshold, grazing=grazing,
                                     sample_mode="bilinear", two_sided_tau=two_sided_tau, return_detail=True)
    u, v, z, dot = det["u"], det["v"], det["z"], det["dot"]
    own = src_view == t
    tie = (np.abs(u) < EPS_PX) | (np.abs(u - w) < EPS_PX) | (np.abs(v) < EPS_PX) | (np.abs(v - h) < EPS_PX)
    tie |= np.abs(z) < EPS_Z
    tie |= np.abs(dot - grazing) < EPS_DOT
    cand = det["inb"] & ~own
    thr32 = np.float32(depth_threshold)

    def decide(x0, y0):
        """decision and near-threshold flag when the sample cell is (x0, y0) (weights from the true u, v)."""
        ok = cand & (x0 >= 0) & (x0 < w) & (y0 >= 0) & (y0 < h)
        x0c, y0c = np.clip(x0, 0, w - 1), np.clip(y0, 0, h - 1)
        x1c, y1c = np.clip(x0 + 1, 0, w - 1), np.clip(y0 + 1, 0, h - 1)
        taps = np.stack([refined_t[y0c, x0c], refined_t[y0c, x1c], refined_t[y1c, x0c], refined_t[y1c, x1c]]).astype(np.float64)
        fx, fy = u - x0, v - y0
        D = (1 - fx) * (1 - fy) * taps[0] + fx * (1 - fy) * taps[1] + (1 - fx) * fy * taps[2] + fx * fy * taps[3]
        valid = ok & (taps > 0).all(0)
        band = EPS_REL * np.abs(D) + EPS_PX * 2 * (taps.max(0) - taps.min(0))
        if two_sided_tau is None:
            q = z - thr32 * D
            dec = valid & (q < 0)
        else:
            q = np.abs(z - D) - np.float32(two_sided_tau) * D
            dec = valid & (q > 0)
        return dec, valid & (np.abs(q) < band)

    x0 = np.floor(np.where(cand, u, 0)).astype(int)
    y0 = np.floor(np.where(cand, v, 0)).astype(int)
    base, near = decide(x0, y0)
    tie |= near
    fu, fv = u - np.floor(u), v - np.floor(v)
    for du, dv, sel in (
        (-1, 0, fu < EPS_PX), (1, 0, fu > 1 - EPS_PX), (0, -1, fv < EPS_PX), (0, 1, fv > 1 - EPS_PX),
        (-1, -1, (fu < EPS_PX) & (fv < EPS_PX)), (1, 1, (fu > 1 - EPS_PX) & (fv > 1 - EPS_PX)),
        (-1, 1, (fu < EPS_PX) & (fv > 1 - EPS_PX)), (1, -1, (fu > 1 - EPS_PX) & (fv < EPS_PX)),
    ):
        sel = sel & cand
        if sel.any():
            alt, near_alt = decide(x0 + du, y0 + dv)
            tie |= sel & ((alt != base) | near_alt)
    # own view: it reprojects to u = x*d/(d+1e-8), a hair below the pixel itself, so the sample is the pixel's own
    # depth up to a relative weight of x*1e-8/d on its neighbours and neither test can fire (K4 skips these pairs).
    # A pair only differs from K4's "no vote" where the statement votes after all.
    tie = np.where(own, vote, tie)
    return vote, tie


def votes_with_ties(points, normals, src_view, refined_all, poses, intr, nbr, active=None, sample_mode="nearest", **kw):
    """Oracle votes[N] and the number of tie pairs per point, honouring the neighbour table."""
    V = refined_all.shape[0]
    votes = np.zeros(len(points), dtype=np.int64)
    nties = np.zeros(len(points), dtype=np.int64)
    member = np.zeros((V, V), dtype=bool)
    for s in range(V):
        for t in nbr[s]:
            if t >= 0:
                member[s, t] = True
    for t in range(V):
        if active is not None and t not in active:
            continue
        sel = np.where(member[src_view, t])[0]
        if len(sel) == 0:
            continue
        fn = pair_ties if sample_mode == "nearest" else pair_ties_bilinear
        vt, tt = fn(points[sel], normals[sel], src_view[sel], t, refined_all[t], poses[t], intr[t], **kw)
        votes[sel] += vt
        nties[sel] += tt
    return votes, nties


def own_view_votes(points, normals, src_view, refined_all, poses, intr, **kw):
    """Number of points the statement's own view votes against (pair_ties_bilinear counts each as a tie)."""
    n = 0
    for s in np.unique(src_view):
        sel = np.where(src_view == s)[0]
        n += int(R.votes_against_view(points[sel], normals[sel], refined_all[s], poses[s], intr[s], **kw).sum())
    return n


def assert_votes_match(gpu_votes, ref_votes, nties, max_tie_fraction=0.02):
    gpu_votes = np.asarray(gpu_votes, dtype=np.int64)
    clean = nties == 0
    bad = clean & (gpu_votes != ref_votes)
    assert not bad.any(), f"{bad.sum()} of {clean.sum()} tie-free points differ; first {np.where(bad)[0][:5]}"
    diff = np.abs(gpu_votes - ref_votes)
    assert (diff <= nties).all(), "vote difference exceeds the number of tie pairs"
    frac = 1.0 - clean.mean() if len(clean) else 0.0
    assert frac <= max_tie_fraction, f"tie fraction {frac:.4f} too large for a meaningful test"
    return frac
