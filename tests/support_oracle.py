"""The multi-view support test (parity unpinned: no reference implementation) and its keep rule, restated on the host.

Built only from oracle/restatement.py's per-view functions, like tests/ragged_oracle.py.  For a point of source view s
and a neighbour entry t of the table: project the point exactly as ``votes_against_view`` does ((u, v, z) in float64,
in bounds iff 0 <= u < W_t, 0 <= v < H_t and z > 0), sample D the way ``sample_mode`` says (truncation; or four taps,
all > 0), and t SUPPORTS the point iff it is in bounds, D > 0 and |z - D| <= float32(tau) * D.  No grazing gate.
Entries of the source view itself and -1 padding never count; a view listed twice counts twice, as the device tests
every entry of the table."""

from __future__ import annotations

import numpy as np

from oracle import restatement as R


def support_of_view(points, refined_t, cam_from_world_t, intr_t, support_tau=0.01, sample_mode="nearest"):
    """bool per point: view t supports it (arguments as ``R.votes_against_view``)."""
    n = len(points)
    _, det = R.votes_against_view(points, np.zeros((n, 3)), refined_t, cam_from_world_t, intr_t, grazing=-np.inf,
                                  sample_mode=sample_mode, return_detail=True)
    if "D" not in det:  # nothing in bounds
        return np.zeros(n, dtype=bool)
    inb, z, D = det["inb"], det["z"], det["D"]
    ok = inb & (D > 0)
    if sample_mode != "nearest":  # all four taps > 0 (a zero tap can leave a positive weighted sum)
        h, w = refined_t.shape
        x0 = np.floor(np.where(inb, det["u"], 0)).astype(int)
        y0 = np.floor(np.where(inb, det["v"], 0)).astype(int)
        x1, y1 = np.clip(x0 + 1, 0, w - 1), np.clip(y0 + 1, 0, h - 1)
        x0, y0 = np.clip(x0, 0, w - 1), np.clip(y0, 0, h - 1)
        ok &= (refined_t[y0, x0] > 0) & (refined_t[y0, x1] > 0) & (refined_t[y1, x0] > 0) & (refined_t[y1, x1] > 0)
    return ok & (np.abs(z - D) <= np.float32(support_tau) * D)


def table_multiplicity(nbr, V):
    """mult[s, t]: how many entries of row s of the table are view t != s."""
    mult = np.zeros((V, V), dtype=np.int64)
    for s in range(V):
        for t in nbr[s]:
            if 0 <= t < V and t != s:
                mult[s, t] += 1
    return mult


def consistency_support(points, src_view, refined_all, poses, intr, nbr, view_ids=None, support_tau=0.01,
                        sample_mode="nearest"):
    """Supporting entries of every point among the table row of its source view (int64, not saturated).
    ``refined_all``: [V,H,W] array or a list of V maps of their own sizes."""
    V = len(refined_all)
    mult = table_multiplicity(nbr, V)
    support = np.zeros(len(points), dtype=np.int64)
    for t in range(V):
        if view_ids is not None and t not in view_ids:
            continue
        sel = np.where(mult[src_view, t] > 0)[0]
        if len(sel) == 0:
            continue
        ok = support_of_view(points[sel], refined_all[t], poses[t], intr[t], support_tau, sample_mode)
        support[sel] += ok * mult[src_view[sel], t]
    return support


def keep(votes, support, vote_threshold, min_support):
    """The keep rule: votes below the threshold (any count at a threshold of 255 or more, as the device clamps it) and
    at least min_support supporting entries."""
    return ((votes < vote_threshold) | (vote_threshold >= 255)) & (support >= min_support)


def encode_votes(votes, support, vote_threshold, min_support):
    """The vote byte the device stores for each point (include/ddn_b200.h, ddn_backproject_filter_support)."""
    cap = 253 if vote_threshold >= 255 else 254
    return np.where(support < min_support, 254, np.minimum(votes, cap)).astype(np.uint8)


def support_bytes(support):
    return np.minimum(support, 254).astype(np.uint8)


# Tie bands, the ones tests/parity.py states for the vote: the device projects in float32 with u = U / Z (no +1e-8), so
# a point within EPS_PX of a map border, or of an integer u or v where the neighbouring pixel (nearest) or cell
# (bilinear) would change the decision, may fall on either side; so may a point within EPS_REL * D of the support
# boundary |z - D| = tau * D (bilinear: plus EPS_PX * 2 * (largest - smallest tap), the sub-pixel error times the slope).
from parity import EPS_PX, EPS_REL, EPS_Z  # noqa: E402


def pair_support_ties(points, refined_t, pose_t, intr_t, support_tau=0.01, sample_mode="nearest"):
    """(support[N] bool, tie[N] bool) of all points against neighbour view t."""
    h, w = refined_t.shape
    n = len(points)
    _, det = R.votes_against_view(points, np.zeros((n, 3)), refined_t, pose_t, intr_t, grazing=-np.inf,
                                  sample_mode=sample_mode, return_detail=True)
    u, v, z, inb = det["u"], det["v"], det["z"], det["inb"]
    tau32 = np.float32(support_tau)
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
        return valid & (q <= 0), valid & (np.abs(q) < band)

    x0 = np.floor(np.where(inb, u, 0)).astype(int)
    y0 = np.floor(np.where(inb, v, 0)).astype(int)
    base, near = decide(x0, y0)
    tie |= near
    fu, fv = u - np.floor(u), v - np.floor(v)
    for du, dv, sel in (
        (-1, 0, fu < EPS_PX), (1, 0, fu > 1 - EPS_PX), (0, -1, fv < EPS_PX), (0, 1, fv > 1 - EPS_PX),
        (-1, -1, (fu < EPS_PX) & (fv < EPS_PX)), (1, 1, (fu > 1 - EPS_PX) & (fv > 1 - EPS_PX)),
        (-1, 1, (fu < EPS_PX) & (fv > 1 - EPS_PX)), (1, -1, (fu > 1 - EPS_PX) & (fv < EPS_PX)),
    ):
        sel = sel & inb
        if sel.any():
            alt, near_alt = decide(x0 + du, y0 + dv)
            tie |= sel & ((alt != base) | near_alt)
    return support_of_view(points, refined_t, pose_t, intr_t, support_tau, sample_mode), tie


def support_with_ties(points, src_view, refined_all, poses, intr, nbr, support_tau=0.01, sample_mode="nearest"):
    """(support[N] int64, ties[N] int64, pair tie fraction): the count of ``consistency_support``, the number of entries
    per point whose decision lies inside a tie band, and the share of all tested (point, entry) pairs that do."""
    V = len(refined_all)
    mult = table_multiplicity(nbr, V)
    support = np.zeros(len(points), dtype=np.int64)
    ties = np.zeros(len(points), dtype=np.int64)
    pairs = 0
    for t in range(V):
        sel = np.where(mult[src_view, t] > 0)[0]
        if len(sel) == 0:
            continue
        ok, tie = pair_support_ties(points[sel], refined_all[t], poses[t], intr[t], support_tau, sample_mode)
        w = mult[src_view[sel], t]
        support[sel] += ok * w
        ties[sel] += tie * w
        pairs += int(w.sum())
    return support, ties, float(ties.sum()) / max(pairs, 1)
