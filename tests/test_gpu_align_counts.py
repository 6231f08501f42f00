"""Stage 1 (align_stats_kernel + remap_median_kernel) at real sparse-point counts, in every workspace placement.

plan_align places a call's buffers by its bound C = max_sparse_per_view, the largest count of any view in the call:
the sort buffer (Cp = next power of two >= C u64 entries) in shared memory up to kSortSmemMax entries, the five pair
arrays (zd, zc, ratio, tx, ty) next to it while Cp * 8 + 20 C fits the pair budget, K3's lookup table in shared memory
(bucketed search) up to kLutSmemMax knots, in global memory (binary search) beyond.  A COLMAP view often sees 5 to 20
thousand points, and one such view moves every view of its call onto the global paths.  Here one scene mixes every
view status with counts on both sides of each placement boundary, the boundaries read from csrc/align.cu; each view
must give the same bits in every placement, and match the oracle (oracle/restatement.py:refine_view) in each
configuration.  At these counts the lookup tables contain knots of equal x and different y, where the result depends on
the tie order (the kernel and the oracle both keep pair order); the unsubsampled comparison asserts that it meets them."""

import re
from dataclasses import dataclass, replace
from pathlib import Path

import numpy as np
import pytest
import torch

from depthdensifier_b200.hashperm import hash_perm
from depthdensifier_b200.neighbours import all_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # refined depth (north_star); affine mode: 2e-5, as test_gpu_parity.test_align_affine_mode
SCALE_RTOL = 2e-6  # scale_factor, as the golden refiner test allows
H, W = 480, 640
N_SPARSE = 24000
REFINED, NO_POINTS_IN_BOUNDS, NO_POSITIVE_SAMPLES, TOO_FEW, NO_SPARSE = 0, 1, 2, 3, 5
ALIGN_CU = Path(__file__).resolve().parent.parent / "depthdensifier_b200" / "csrc" / "align.cu"


@dataclass(frozen=True)
class Thresholds:
    sort: int  # kSortSmemMax: u64 sort entries in shared memory
    pair_bytes: int  # shared memory for the sort buffer and the pair arrays together
    lut: int  # kLutSmemMax: lookup-table knots in shared memory


def _thresholds() -> Thresholds:
    src = ALIGN_CU.read_text()

    def find(pattern):
        m = re.search(pattern, src)
        assert m, f"{pattern!r} not found in {ALIGN_CU.name}"
        return int(m.group(1))

    return Thresholds(sort=find(r"constexpr int kSortSmemMax = (\d+);"),
                      pair_bytes=find(r"p\.ws\.Cp \* 8 \+ \(size_t\)p\.ws\.C \* 20 <= (\d+) \* 1024") * 1024,
                      lut=find(r"constexpr int kLutSmemMax = (\d+);"))


def _placement(C: int, opts, T: Thresholds):
    """plan_align's choice for bound C: (sort buffer in shared memory, pair arrays in shared memory, lookup table in
    shared memory, Cp)."""
    Cp = 2
    while Cp < C:
        Cp *= 2
    sort = Cp <= T.sort
    pairs = sort and Cp * 8 + 20 * C <= T.pair_bytes
    knots = opts.max_pairs if opts.adaptive_correspondences and opts.max_pairs < C else C
    return sort, pairs, opts.align_mode == "pwl" and knots <= T.lut, Cp


def _boundaries(T: Thresholds) -> list:
    """Counts C at which the placement of an unsubsampled call differs at C + 1, from the table's size on (smaller
    bounds only resize the shared buffers) to the end of the shared sort: 4096 (table, Cp), 6963 (pair arrays),
    8192 (Cp) and 16384 (sort buffer) with the thresholds of this writing."""
    from depthdensifier_b200.ops import AlignOptions

    o = AlignOptions(adaptive_correspondences=False)
    end = T.sort  # kSortSmemMax is a power of two: the last bound whose sort buffer fits
    return [C for C in range(T.lut, end + 1) if _placement(C, o, T) != _placement(C + 1, o, T)]


@dataclass
class View:
    kind: str
    depth: np.ndarray  # [H,W] f32
    mask: np.ndarray  # [H,W] bool
    xyz: np.ndarray  # [n,3] f64
    pose: np.ndarray
    kmat: np.ndarray
    intr: np.ndarray


def _project(xyz, pose, intr):
    cam = xyz @ pose[:, :3].T + pose[:, 3]
    return intr[0] * cam[:, 0] / cam[:, 2] + intr[2], intr[1] * cam[:, 1] / cam[:, 2] + intr[3], cam


@pytest.fixture(scope="module")
def scene():
    """One view per status and per count on each side of every placement boundary, one view of at least 20k points
    and one whose mono depth is quantised to millimetres (as 16-bit depth files store it)."""
    T = _thresholds()
    bounds = _boundaries(T)
    counts = [("no_sparse", 0), ("behind_camera", 300), ("zero_depth", 200), ("too_few", 30), ("small", 300)]
    counts += [(f"count_{c}", c) for b in bounds for c in (b, b + 1)]
    counts += [("large", N_SPARSE), ("millimetres", 20000)]
    sc = make_scene(SceneConfig(n_views=len(counts), width=W, height=H, n_sparse=N_SPARSE, seed=7))
    off = sc.sparse_offsets.numpy()
    views = []
    for v, (kind, n) in enumerate(counts):
        pose, intr = sc.cam_from_world[v].numpy(), sc.intrinsics[v].numpy()
        depth, mask = sc.mono_depth[v].numpy().copy(), sc.mask[v].numpy()
        pts = sc.sparse_xyz[off[v]:off[v + 1]].numpy()
        assert len(pts) == N_SPARSE
        if kind == "behind_camera":  # mirrored through the image plane: z_cam < 0 for all
            cam = pts[:n] @ pose[:, :3].T + pose[:, 3]
            cam[:, 2] = -np.abs(cam[:, 2]) - 1
            pts = (cam - pose[:, 3]) @ pose[:, :3]
        elif kind == "zero_depth":  # mono depth zeroed in a rectangle; points whose four bilinear taps all lie inside
            y0, y1, x0, x1 = 140, 340, 170, 470
            depth[y0:y1, x0:x1] = 0
            u, w, cam = _project(pts, pose, intr)
            inside = (cam[:, 2] > 0) & (u >= x0 + 2) & (u < x1 - 3) & (w >= y0 + 2) & (w < y1 - 3)
            pts = pts[inside][:n]
            assert len(pts) == n
        else:
            pts = pts[:n]
        if kind == "millimetres":
            depth = (np.round(depth.astype(np.float64) * 1000) / 1000).astype(np.float32)
        views.append(View(kind, depth, mask, np.ascontiguousarray(pts), pose, R.kmatrix(intr), intr))
    return T, bounds, views


def _subsets(views, bounds, T):
    """(view indices, bounds to run them at): the views of at most b points for each boundary b (and all views), at
    their true maximum, at the first bound of every later placement and at 2 kSortSmemMax + 1 (a global sort buffer
    of four times the shared one)."""
    counts = np.array([len(v.xyz) for v in views])
    largest = 2 * T.sort + 1
    out = []
    for b in bounds + [None]:
        idx = np.flatnonzero(counts <= b) if b is not None else np.arange(len(views))
        top = int(counts[idx].max())
        runs = [top] + [c + 1 for c in bounds if c + 1 > top] + [largest]
        out.append((idx, sorted(set(runs))))
    return out


def _inputs(views, idx, mask_on=True):
    cuda = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    sel = [views[i] for i in idx]
    off = np.concatenate([[0], np.cumsum([len(v.xyz) for v in sel])]).astype(np.int64)
    xyz = np.concatenate([v.xyz for v in sel]) if off[-1] else np.zeros((0, 3))
    return dict(depth=cuda(np.stack([v.depth for v in sel])), mask=cuda(np.stack([v.mask for v in sel])) if mask_on else None,
                pose=cuda(np.stack([v.pose for v in sel])), kmat=cuda(np.stack([v.kmat for v in sel])),
                intr=cuda(np.stack([v.intr for v in sel])), sparse=cuda(xyz.astype(np.float64)), off=cuda(off))


def _align(inp, bound, opts, mask="bool", **kw):
    from depthdensifier_b200 import ops

    m = inp["mask"]
    if m is not None and mask == "packed":
        m = ops.pack_mask(m.cpu()).cuda()
    refined, stats = ops.align_views(inp["depth"], m, inp["pose"], inp["kmat"], inp["sparse"], inp["off"], bound, opts, **kw)
    torch.cuda.synchronize()
    return refined, stats


def _oracle_view(view, acfg: R.AlignConfig, mask_on: bool):
    """The oracle's statement of one view in the kernel's terms: status, counts, scale and refined depth."""
    if len(view.xyz) == 0:  # the pipeline skips the view; the kernel writes zeros
        return dict(status=NO_SPARSE, num=0, removed=0, num_table=0, scale=1.0, refined=np.zeros_like(view.depth))

    def run(cfg):
        return R.refine_view(view.depth.copy(), view.xyz, view.pose, view.kmat, view.mask if mask_on else None, cfg,
                             randperm=lambda n: hash_perm(n, 0))

    r = run(acfg)
    num = r["num_correspondences"]
    if "outliers_removed" in r:
        status, removed = REFINED, r["outliers_removed"]
    elif num > 0:  # too few pairs after the IQR step; the kernel still reports what that step removed
        status, removed = TOO_FEW, run(replace(acfg, min_correspondences=0))["outliers_removed"]
    else:
        uv, z = R.project_sparse(torch.from_numpy(view.xyz).float(), torch.from_numpy(view.pose).float(),
                                 torch.from_numpy(view.kmat).float())
        m = acfg.edge_margin
        inb = (uv[:, 0] >= m) & (uv[:, 0] < W - m) & (uv[:, 1] >= m) & (uv[:, 1] < H - m) & (z > 0)
        status, removed = (NO_POSITIVE_SAMPLES if bool(inb.any()) else NO_POINTS_IN_BOUNDS), 0
    return dict(status=status, num=num, removed=removed, scale=r["scale_factor"], refined=np.asarray(r["refined_depth"], np.float32),
                num_table=num if status == REFINED and acfg.align_mode == "pwl" else 0)


CONFIGS = {
    "default": dict(),
    "no_subsample": dict(adaptive_correspondences=False),
    "not_robust": dict(adaptive_correspondences=False, robust=False),
    "skip_smoothing": dict(adaptive_correspondences=False, skip_smoothing=True),
    "max_pairs_5000": dict(max_pairs=5000),
    "affine": dict(align_mode="affine"),
    "mask_none": dict(adaptive_correspondences=False),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_align_placements_and_oracle(lib_built, scene, name, monkeypatch):
    from depthdensifier_b200 import ops

    T, bounds, views = scene
    kw = CONFIGS[name]
    mask_on = name != "mask_none"
    opts = ops.AlignOptions(**kw)

    # placement invariance: every view gives the same bits in every call that contains it
    first, placements = {}, set()
    for idx, runs in _subsets(views, bounds, T):
        inp = _inputs(views, idx, mask_on)
        for bound in runs:
            placements.add(_placement(bound, opts, T))
            refined, stats = _align(inp, bound, opts)
            for j, v in enumerate(idx):
                got = (refined[j].view(torch.int32), stats[j])
                if v not in first:
                    first[v] = got
                else:
                    assert torch.equal(first[v][1], got[1]), (name, views[v].kind, bound, ops.decode_stats(got[1][None]))
                    assert torch.equal(first[v][0], got[0]), (name, views[v].kind, bound)
    rows = {p[:3] for p in placements}
    assert {(True, True), (True, False), (False, False)} <= {r[:2] for r in rows}, rows  # sort / pair placements
    for b in bounds:  # both sides of every boundary
        assert _placement(b, opts, T) in placements and _placement(b + 1, opts, T) in placements, (b, placements)
    if opts.align_mode == "pwl" and not opts.adaptive_correspondences:
        assert {True, False} <= {r[2] for r in rows}, rows  # both K3 lookup forms
    print(f"\n[{name}] placements (sort smem, pairs smem, table smem, Cp): {sorted(placements)}")

    # against the oracle, view by view; the oracle's lookup tables are recorded on the way
    tables, fits = [], []
    pwl_lookup, affine_fit = R.pwl_lookup, R.affine_fit

    def record_lookup(d, x, y):
        out = pwl_lookup(d, x, y)
        xn, yn = x.numpy(), y.numpy()
        u, c = np.unique(xn, return_counts=True)
        differ = sum(len(np.unique(yn[xn == r])) > 1 for r in u[c > 1])
        # the same table with equal knots in reverse pair order: the pixels whose value the tie order decides
        swapped = int((pwl_lookup(d, x.flip(0), y.flip(0)) != out).sum())
        tables.append((differ, swapped))
        return out

    def record_fit(d, z):
        fits.append(affine_fit(d, z))
        return fits[-1]

    monkeypatch.setattr(R, "pwl_lookup", record_lookup)
    monkeypatch.setattr(R, "affine_fit", record_fit)
    acfg = R.AlignConfig(**kw)
    stats_all = ops.decode_stats(torch.stack([first[v][1] for v in range(len(views))]))
    statuses = []
    for v, view in enumerate(views):
        n_tables, n_fits = len(tables), len(fits)
        ref = _oracle_view(view, acfg, mask_on)
        st, got = stats_all[v], first[v][0].view(torch.float32).cpu().numpy()
        where = (name, view.kind, len(view.xyz))
        statuses.append(st["status"])
        assert st["status"] == ref["status"], (where, st)
        assert st["num_correspondences"] == ref["num"], (where, st, ref["num"])
        assert st["outliers_removed"] == ref["removed"], (where, st, ref["removed"])
        assert st["num_table"] == ref["num_table"], (where, st)
        assert abs(st["scale_factor"] - ref["scale"]) <= SCALE_RTOL * abs(ref["scale"]), (where, st, ref["scale"])
        assert np.array_equal(got == 0, ref["refined"] == 0), where
        np.testing.assert_allclose(got, ref["refined"], rtol=2e-5 if opts.align_mode == "affine" else RTOL, atol=0, err_msg=str(where))
        if opts.align_mode == "affine" and ref["status"] == REFINED:
            s, t = fits[n_fits]
            np.testing.assert_allclose([st["affine_scale"], st["affine_shift"]], [s, t], rtol=2e-5, atol=2e-5 * abs(s), err_msg=str(where))
        if view.kind == "millimetres" and not opts.adaptive_correspondences and opts.align_mode == "pwl":
            assert tables[n_tables][0] > 0 and tables[n_tables][1] > 0, tables[n_tables]  # the quantised view has ties
    assert set(statuses) == {REFINED, NO_POINTS_IN_BOUNDS, NO_POSITIVE_SAMPLES, TOO_FEW, NO_SPARSE}, statuses
    print(f"[{name}] statuses by view: {dict(zip([v.kind for v in views], statuses))}")
    if tables:
        print(f"[{name}] knots of equal x and different y: {sum(t[0] for t in tables)} over {len(tables)} tables; "
              f"pixels decided by the tie order: {sum(t[1] for t in tables)}")
    if name == "no_subsample":  # full-size tables: the comparison above met the tie case
        assert sum(t[0] for t in tables) > 0 and sum(t[1] for t in tables) > 0, tables


@pytest.mark.parametrize("name", ["default", "no_subsample"])
def test_remap_forms_at_global_placements(lib_built, scene, name):
    """The bit-packed mask, the TMA tile load, the ragged entry point and the bounding-box epilogue at the largest bound
    give the default call's bits; the box is the same whichever form computes it, at any bound, and encloses every
    back-projected refined pixel."""
    from depthdensifier_b200 import ops

    T, bounds, views = scene
    idx = np.arange(len(views))
    inp = _inputs(views, idx)
    top, largest = max(len(v.xyz) for v in views), 2 * T.sort + 1
    opts = ops.AlignOptions(**CONFIGS[name])
    assert _placement(largest, opts, T)[:2] == (False, False)  # sort buffer and pair arrays in global memory
    base = _align(inp, largest, opts)

    def same(out, what):
        assert torch.equal(out[1], base[1]), what
        assert torch.equal(out[0].reshape(base[0].shape).view(torch.int32), base[0].view(torch.int32)), what

    same(_align(inp, largest, opts, mask="packed"), "packed mask")
    same(_align(inp, largest, replace(opts, use_tma=True)), "use_tma")
    layout = ops.ViewLayout([(H, W)] * len(views))
    V = len(views)

    def ragged(bound, **kw):
        out = ops.align_views_ragged(layout, inp["depth"].reshape(-1), inp["mask"].reshape(-1), inp["pose"], inp["kmat"], inp["sparse"],
                                     inp["off"], bound, opts, **kw)
        torch.cuda.synchronize()
        return out

    same(ragged(largest), "ragged")
    nbr = torch.from_numpy(all_views_table(V).astype(np.int32)).cuda()
    _, src = ops.build_pair_tables(inp["pose"], inp["intr"], nbr, 0, V, H, W)
    _, src_r = ops.build_pair_tables_ragged(layout, inp["pose"], inp["intr"], nbr)
    boxes = []
    for bound in (top, largest):
        bbox = ops.new_bbox(inp["depth"].device)
        same(_align(inp, bound, opts, src_table=src, bbox=bbox), f"bbox epilogue at {bound}")
        boxes.append(ops.decode_bbox(bbox))
        bbox = ops.new_bbox(inp["depth"].device)
        same(ragged(bound, src_table=src_r, bbox=bbox), f"ragged bbox epilogue at {bound}")
        boxes.append(ops.decode_bbox(bbox))
    assert all(np.array_equal(b, boxes[0]) for b in boxes[1:]), boxes
    refined = base[0].cpu().numpy()
    pts = np.concatenate([R.backproject_view(refined[v], views[v].intr, views[v].pose)[0] for v in range(V)])
    assert len(pts) > 0
    slack = 1e-5 * max(1.0, np.abs(pts).max())
    assert (pts.min(0) >= boxes[0][:3] - slack).all() and (pts.max(0) <= boxes[0][3:] + slack).all(), (pts.min(0), pts.max(0), boxes[0])
