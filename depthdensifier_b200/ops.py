"""Device-tensor wrappers around the C ABI.  torch is plumbing only (device memory + streams); every
op below runs a hand-written sm_100a kernel from libddn_b200.so and raises when no GPU is present."""

from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._lib import DDNError

STATUS_REFINED = 0
STATUS_NAMES = {
    0: "refined",
    1: "no_points_in_bounds",
    2: "no_positive_samples",
    3: "too_few_correspondences",
    4: "degenerate_fit",
    5: "no_sparse_points",
}


def _require_cuda(*tensors) -> torch.device:
    if not torch.cuda.is_available():
        raise DDNError("no CUDA device available: depthdensifier_b200 has no CPU fallback")
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise DDNError("expected CUDA tensors")
        if not t.is_contiguous():
            raise DDNError("expected contiguous tensors")
        dev = t.device if dev is None else dev
        if t.device != dev:
            raise DDNError("tensors on different devices")
    return dev


def _require_cuda_normal(normal, *tensors) -> torch.device:
    """_require_cuda for the consistency kernel's inputs: ``normal`` may also be a pinned host tensor."""
    normal_on_host = not normal.is_cuda
    if normal_on_host and not (normal.is_pinned() and normal.is_contiguous()):
        raise DDNError("a host normal map must be pinned and contiguous")
    return _require_cuda(None if normal_on_host else normal, *tensors)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@dataclass
class AlignOptions:
    """RefinerConfig fields (depth_refiner.py:16-31) + the north-star mode switch."""

    min_correspondences: int = 50
    edge_margin: int = 10
    robust: bool = True
    outlier_threshold: float = 2.5
    skip_smoothing: bool = False
    adaptive_correspondences: bool = True
    max_pairs: int = 500
    align_mode: str = "pwl"
    subsample_seed: int = 0
    zero_unmasked_passthrough: bool = False
    use_tma: bool = False  # K3 depth tile via one TMA tensor copy (W % 4 == 0, W >= 132, H >= 34): same bits, measured 6 % slower

    def to_c(self, mask_packed: bool = False) -> _lib.AlignConfig:
        if self.align_mode not in ("pwl", "affine"):
            raise ValueError("align_mode must be 'pwl' or 'affine'")
        return _lib.AlignConfig(
            int(self.min_correspondences),
            int(self.edge_margin),
            int(bool(self.robust)),
            float(self.outlier_threshold),
            int(bool(self.skip_smoothing)),
            int(bool(self.adaptive_correspondences)),
            int(self.max_pairs),
            0 if self.align_mode == "pwl" else 1,
            int(self.subsample_seed) & 0xFFFFFFFF,
            int(bool(self.zero_unmasked_passthrough)),
            int(bool(mask_packed)),
            int(bool(self.use_tma)),
        )


@dataclass
class FilterOptions:
    depth_threshold: float = 0.7
    grazing_cos: float = 0.087
    sample_mode: str = "nearest"
    two_sided_tau: float = 0.0
    stride: int = 1
    normals_in_world: bool = False
    pixel_layout: int = 0  # which 4 pixels a K4 thread owns: 0 = 32 apart, 1 = adjacent (same results)

    def to_c(self) -> _lib.FilterConfig:
        if self.sample_mode not in ("nearest", "bilinear"):
            raise ValueError("sample_mode must be 'nearest' or 'bilinear'")
        return _lib.FilterConfig(
            float(self.depth_threshold),
            float(self.grazing_cos),
            0 if self.sample_mode == "nearest" else 1,
            float(self.two_sided_tau),
            int(self.stride),
            int(bool(self.normals_in_world)),
            int(self.pixel_layout),
        )


def intrinsics_matrix(intr) -> torch.Tensor:
    """[V,3,3] f64 camera matrices from PINHOLE intrinsics [V,4] = (fx, fy, cx, cy)."""
    kmat = torch.zeros((intr.shape[0], 3, 3), dtype=torch.float64, device=intr.device)
    kmat[:, 0, 0], kmat[:, 1, 1], kmat[:, 0, 2], kmat[:, 1, 2], kmat[:, 2, 2] = intr[:, 0], intr[:, 1], intr[:, 2], intr[:, 3], 1.0
    return kmat


def _align_scratch(lib, n_views: int, max_sparse_per_view: int, dev):
    """The zeroed stats [V,8] and the workspace (tensor, bytes) of one alignment call."""
    stats = torch.zeros((n_views, 8), dtype=torch.int32, device=dev)
    nbytes = C.c_int64(0)
    _lib.check(lib.ddn_align_workspace_bytes(n_views, max_sparse_per_view, C.byref(nbytes)))
    return stats, torch.empty(nbytes.value, dtype=torch.uint8, device=dev), nbytes.value


def align_views(depth, mask, cam_from_world, kmat, sparse_xyz, sparse_offsets, max_sparse_per_view: int,
                opts: AlignOptions, out=None, src_table=None, bbox=None):
    """Stage 1 for V views.  Returns (refined [V,H,W] f32, stats [V,8] int32 raw ddn_view_stats).
    ``src_table`` [V,16] (from build_pair_tables) + ``bbox`` [6] (new_bbox): the kernel also extends the box to
    enclose the back-projection of every refined pixel, so the voxel grid is known before stages 2+3."""
    lib = _lib.load()
    dev = _require_cuda(depth, mask, cam_from_world, kmat, sparse_xyz, sparse_offsets, out, src_table, bbox)
    assert (src_table is None) == (bbox is None)
    assert src_table is None or (src_table.dtype == torch.float32 and tuple(src_table.shape) == (depth.shape[0], 16))
    V, H, W = depth.shape
    assert depth.dtype == torch.float32 and cam_from_world.dtype == torch.float64 and kmat.dtype == torch.float64
    assert sparse_xyz.dtype == torch.float64 and sparse_offsets.dtype == torch.int64
    # a 2-D uint8 mask [V, ceil(H*W/8)] is the bit-packed form (pack_mask)
    packed = mask is not None and mask.dtype == torch.uint8 and mask.dim() == 2
    assert mask is None or (packed and tuple(mask.shape) == (V, (H * W + 7) // 8)) or (
        mask.dtype in (torch.bool, torch.uint8) and mask.shape == depth.shape)
    assert tuple(cam_from_world.shape) == (V, 3, 4) and tuple(kmat.shape) == (V, 3, 3)
    refined = out if out is not None else torch.empty_like(depth)
    stats, ws, nbytes = _align_scratch(lib, V, max_sparse_per_view, dev)
    cfg = opts.to_c(mask_packed=packed)
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_align_views(
                C.byref(cfg), V, H, W, _p(depth), _p(mask), _p(cam_from_world), _p(kmat), _p(sparse_xyz),
                _p(sparse_offsets), int(max_sparse_per_view), _p(refined), _p(stats), _p(ws), nbytes, _p(src_table),
                _p(bbox), _stream(),
            )
        )
    return refined, stats


def pack_mask(mask: torch.Tensor) -> torch.Tensor:
    """[V,H,W] bool mask -> [V, ceil(H*W/8)] uint8, one bit per pixel (bit g & 7 of byte g >> 3): the form the alignment
    kernel also accepts, an eighth of the bytes to upload.  Host tensors (numpy packbits)."""
    m = np.ascontiguousarray(mask.cpu().numpy()).reshape(mask.shape[0], -1)
    return torch.from_numpy(np.packbits(m, axis=1, bitorder="little"))


def decode_stats(stats: torch.Tensor) -> list[dict]:
    """Host dicts from the raw [V,8] int32 stats tensor (synchronises)."""
    s = stats.cpu().numpy()
    f = s.view(np.float32)
    out = []
    for v in range(s.shape[0]):
        out.append(
            {
                "status": int(s[v, 0]),
                "num_correspondences": int(s[v, 1]),
                "outliers_removed": int(s[v, 2]),
                "num_table": int(s[v, 3]),
                "scale_factor": float(f[v, 4]),
                "affine_scale": float(f[v, 5]),
                "affine_shift": float(f[v, 6]),
            }
        )
    return out


def build_pair_tables(cam_from_world, intr, nbr, src_begin: int, n_src: int, height: int, width: int):
    """Per-(source view, neighbour) float32 tables from the float64 poses; ``height`` / ``width``: the size of the
    depth maps the tables will be used with (K4's gather offsets are precomputed per entry)."""
    lib = _lib.load()
    dev = _require_cuda(cam_from_world, intr, nbr)
    V = cam_from_world.shape[0]
    K = nbr.shape[1]
    assert cam_from_world.dtype == torch.float64 and intr.dtype == torch.float64 and nbr.dtype == torch.int32
    assert tuple(intr.shape) == (V, 4) and nbr.shape[0] == V
    pair = torch.empty((n_src, K, _lib.PAIR_TABLE_FLOATS), dtype=torch.float32, device=dev)
    src = torch.empty((n_src, 16), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_build_pair_tables(V, src_begin, n_src, K, int(height), int(width), _p(cam_from_world), _p(intr), _p(nbr),
                                             _p(pair), _p(src), _stream()))
    return pair, src


def init_bbox(bbox: torch.Tensor) -> torch.Tensor:
    """(+inf, -inf) in the order-preserving int encoding the kernels fold points into."""
    lib = _lib.load()
    with torch.cuda.device(bbox.device):
        _lib.check(lib.ddn_bbox_init(_p(bbox), _stream()))
    return bbox


def new_bbox(dev) -> torch.Tensor:
    return init_bbox(torch.empty(6, dtype=torch.int32, device=dev))


def decode_bbox(bbox: torch.Tensor) -> np.ndarray:
    """[6] float32 (min xyz, max xyz) from the order-preserving int encoding (synchronises)."""
    i = bbox.cpu().numpy().astype(np.int32)
    i = np.where(i >= 0, i, i ^ np.int32(0x7FFFFFFF))
    return i.view(np.float32)


def _support_args(support) -> tuple[int, float, float | None]:
    """(min_support, tau, reproj_px or None) from ``support`` = (m, tau) or (m, tau, reproj_px)."""
    if len(support) not in (2, 3):
        raise ValueError(f"support = (min_support, tau) or (min_support, tau, reproj_px), got {support}")
    m, tau = support[:2]
    if not (0 <= int(m) <= 1024) or not (math.isfinite(float(tau)) and float(tau) > 0):
        raise ValueError(f"support = (min_support in [0, 1024], tau > 0 finite), got {support}")
    rho = None
    if len(support) == 3:
        rho = float(support[2])
        if not (math.isfinite(rho) and rho > 0):
            raise ValueError(f"support = (min_support, tau, reproj_px > 0 finite), got {support}")
    return int(m), float(tau), rho


def fusion_threshold(vote_threshold: int, support: bool) -> int:
    """The threshold fusion and keep masks test the vote bytes of a filter call with: ``vote_threshold``, or
    min(vote_threshold, 254) when the call counted support (the vote byte then carries the keep decision; see
    ddn_backproject_filter_support in include/ddn_b200.h)."""
    return min(int(vote_threshold), 254) if support else int(vote_threshold)


def backproject_filter(refined_all, normal, nbr, pair_table, src_table, src_begin: int, vote_threshold: int,
                       opts: FilterOptions, bbox=None, xyz_out=None, votes_out=None, mark=None, support=None,
                       support_out=None):
    """Stages 2+3 for the source views src_begin..src_begin+n_src (n_src = normal.shape[0]).  ``normal`` may
    be a PINNED HOST tensor: the kernel then reads the normals of its vote candidates in place over PCIe
    (unified addressing) and the 12 B/pixel normal map never moves to the device.  ``mark``: an open
    ``FuseSession``; the kernel then also sets the occupancy bits of the kept points (stage 4's mark pass).

    ``support`` = (min_support, tau): also count the neighbours that see each point within the relative depth error
    tau and keep only points with at least min_support of them (ddn_backproject_filter_support).  Returns
    (xyz, votes, support) then, support [n_src,Hs,Ws] u8 (or ``support_out``); test the votes with
    ``fusion_threshold(vote_threshold, True)``.  ``support`` = (min_support, tau, reproj_px): a neighbour supports a
    point only when, besides, the round trip source -> neighbour -> source lands within reproj_px pixels of the
    point's pixel (ddn_backproject_filter_support_reproj)."""
    lib = _lib.load()
    dev = _require_cuda_normal(normal, refined_all, nbr, pair_table, src_table, bbox, xyz_out, votes_out)
    V, H, W = refined_all.shape
    n_src = normal.shape[0]
    K = nbr.shape[1]
    assert refined_all.dtype == torch.float32 and normal.dtype == torch.float32
    assert tuple(normal.shape) == (n_src, H, W, 3)
    assert tuple(pair_table.shape) == (n_src, K, _lib.PAIR_TABLE_FLOATS) and tuple(src_table.shape) == (n_src, 16)
    s = int(opts.stride)
    Hs, Ws = (H + s - 1) // s, (W + s - 1) // s
    xyz = xyz_out if xyz_out is not None else torch.empty((n_src, Hs, Ws, 3), dtype=torch.float32, device=dev)
    votes = votes_out if votes_out is not None else torch.empty((n_src, Hs, Ws), dtype=torch.uint8, device=dev)
    cfg = opts.to_c()
    if support is not None:
        m, tau, rho = _support_args(support)
        sup = support_out if support_out is not None else torch.empty((n_src, Hs, Ws), dtype=torch.uint8, device=dev)
        assert sup.dtype == torch.uint8 and sup.is_contiguous() and tuple(sup.shape) == tuple(votes.shape)
        head = (C.byref(cfg), V, src_begin, n_src, H, W, K, _p(refined_all), _p(normal), _p(nbr), _p(pair_table),
                _p(src_table), int(vote_threshold), m, tau)
        tail = (_p(xyz), _p(votes), _p(sup), _p(bbox), C.byref(mark.c) if mark is not None else None, _stream())
        with torch.cuda.device(dev):
            if rho is None:
                _lib.check(lib.ddn_backproject_filter_support(*head, *tail))
            else:
                _lib.check(lib.ddn_backproject_filter_support_reproj(*head, rho, *tail))
        return xyz, votes, sup
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_backproject_filter(
                C.byref(cfg), V, src_begin, n_src, H, W, K, _p(refined_all), _p(normal), _p(nbr), _p(pair_table),
                _p(src_table), int(vote_threshold), _p(xyz), _p(votes), _p(bbox),
                C.byref(mark.c) if mark is not None else None, _stream(),
            )
        )
    return xyz, votes


# ----------------------------------------------------------------------------------------------
# Ragged views: V depth maps of different sizes in one pass (include/ddn_b200.h, DDN_LAYOUT_COLS)
# ----------------------------------------------------------------------------------------------
REMAP_TILE_H, REMAP_TILE_W = 32, 126  # remap_median_kernel tile (align.cu)
FILTER_CHUNK = 1024  # points per consistency-kernel CTA (filter.cu kFilterChunk)
MAX_RAGGED_VIEWS = 65535


class ViewLayout:
    """Sizes and offsets of V views of different sizes concatenated into flat buffers: per-pixel buffers (depth, mask,
    refined, normal, rgb) hold the views' row-major maps one after the other, strided-grid buffers (xyz, votes) their
    ceil(H/stride) x ceil(W/stride) grids.  ``table`` is the int64 [V+1, 8] layout of the C ABI (row v: H, W, pixel
    offset, grid offset, first remap tile, first consistency chunk; last row: stride, V and the four totals)."""

    def __init__(self, shapes, stride: int = 1):
        shapes = [(int(h), int(w)) for h, w in shapes]
        stride = int(stride)
        V = len(shapes)
        if V < 1 or V > MAX_RAGGED_VIEWS:
            raise ValueError(f"a ragged layout holds 1 to {MAX_RAGGED_VIEWS} views, got {V}")
        if stride < 1:
            raise ValueError("stride must be >= 1")
        for h, w in shapes:
            if h < 1 or w < 1:
                raise ValueError(f"zero-sized view {h}x{w}")
            if h >= 1 << 22 or w >= 1 << 22 or h * w >= 1 << 31:
                raise ValueError(f"view {h}x{w} too large (sides < 2^22, fewer than 2^31 pixels)")
        hw = np.array(shapes, dtype=np.int64).reshape(V, 2)
        hs, ws = (hw[:, 0] + stride - 1) // stride, (hw[:, 1] + stride - 1) // stride
        units = np.stack([hw[:, 0] * hw[:, 1], hs * ws,
                          ((hw[:, 0] + REMAP_TILE_H - 1) // REMAP_TILE_H) * ((hw[:, 1] + REMAP_TILE_W - 1) // REMAP_TILE_W),
                          (hs * ws + FILTER_CHUNK - 1) // FILTER_CHUNK], axis=1)
        if units[:, 0].sum() >= 1 << 32:
            raise ValueError(f"{int(units[:, 0].sum())} pixels in all: the ragged kernels address fewer than 2^32")
        t = np.zeros((V + 1, _lib.LAYOUT_COLS), dtype=np.int64)
        t[:V, 0:2] = hw
        t[1:, 2:6] = np.cumsum(units, axis=0)
        t[V, 0:2] = stride, V
        self.shapes, self.stride, self.table = shapes, stride, t
        self.grid_shapes = list(zip(hs.tolist(), ws.tolist()))
        self._dev = {}

    @classmethod
    def from_shapes(cls, shapes, stride: int = 1) -> "ViewLayout":
        return cls(shapes, stride)

    @property
    def n_views(self) -> int:
        return len(self.shapes)

    @property
    def pix_off(self) -> np.ndarray:  # [V+1]
        return self.table[:, 2].copy()

    @property
    def grid_off(self) -> np.ndarray:  # [V+1]
        return self.table[:, 3].copy()

    @property
    def total_pixels(self) -> int:
        return int(self.table[-1, 2])

    @property
    def total_grid(self) -> int:
        return int(self.table[-1, 3])

    @property
    def uniform(self) -> bool:
        return len(set(self.shapes)) == 1

    def device(self, dev) -> torch.Tensor:
        """The layout in device memory (one copy per device, kept)."""
        dev = torch.device(dev)
        if dev not in self._dev:
            self._dev[dev] = torch.from_numpy(self.table).to(dev)
        return self._dev[dev]

    def host_ptr(self):
        return self.table.ctypes.data_as(C.c_void_p)

    def flatten(self, maps, dtype=None) -> torch.Tensor:
        """Concatenation of per-view maps [H_v, W_v, ...] (tensors or arrays, one device) into one flat tensor."""
        ts = [torch.as_tensor(m) for m in maps]
        assert [tuple(t.shape[:2]) for t in ts] == self.shapes, "maps do not match the layout"
        out = torch.cat([t.reshape((-1,) + tuple(t.shape[2:])) for t in ts], 0)
        return out.to(dtype).contiguous() if dtype is not None else out.contiguous()

    def split(self, flat: torch.Tensor, grid: bool = False) -> list:
        """Per-view views [H_v, W_v, ...] (or the strided grids with ``grid``) of a flat tensor; no copy."""
        off = self.table[:, 3 if grid else 2]
        shapes = self.grid_shapes if grid else self.shapes
        return [flat[int(off[v]):int(off[v + 1])].view((h, w) + tuple(flat.shape[1:])) for v, (h, w) in enumerate(shapes)]

    def strided(self, maps) -> list:
        """Each view's map [H_v, W_v, ...] on its strided grid (every stride-th row and column)."""
        s = self.stride
        return [m if s == 1 else m[::s, ::s] for m in maps]


def align_views_ragged(layout: ViewLayout, depth, mask, cam_from_world, kmat, sparse_xyz, sparse_offsets, max_sparse_per_view: int,
                       opts: AlignOptions, out=None, src_table=None, bbox=None):
    """Stage 1 for the views of ``layout``: depth flat [P] f32, mask flat [P] bool/u8 or None, refined flat [P].  Returns
    (refined, stats [V,8]).  ``src_table`` [V,16] + ``bbox`` [6]: the bounding-box epilogue, as in align_views."""
    lib = _lib.load()
    dev = _require_cuda(depth, mask, cam_from_world, kmat, sparse_xyz, sparse_offsets, out, src_table, bbox)
    assert (src_table is None) == (bbox is None)
    V, P = layout.n_views, layout.total_pixels
    assert depth.dtype == torch.float32 and tuple(depth.shape) == (P,)
    assert mask is None or (mask.dtype in (torch.bool, torch.uint8) and tuple(mask.shape) == (P,))
    assert tuple(cam_from_world.shape) == (V, 3, 4) and tuple(kmat.shape) == (V, 3, 3)
    assert sparse_xyz.dtype == torch.float64 and sparse_offsets.dtype == torch.int64
    refined = out if out is not None else torch.empty_like(depth)
    stats, ws, nbytes = _align_scratch(lib, V, max_sparse_per_view, dev)
    cfg = opts.to_c()
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_align_views_ragged(
                C.byref(cfg), V, _p(layout.device(dev)), layout.host_ptr(), _p(depth), _p(mask), _p(cam_from_world), _p(kmat),
                _p(sparse_xyz), _p(sparse_offsets), int(max_sparse_per_view), _p(refined), _p(stats), _p(ws), nbytes,
                _p(src_table), _p(bbox), _stream(),
            )
        )
    return refined, stats


def build_pair_tables_ragged(layout: ViewLayout, cam_from_world, intr, nbr):
    """Pair / source tables for all views of ``layout`` (entries carry the neighbour's own size)."""
    lib = _lib.load()
    dev = _require_cuda(cam_from_world, intr, nbr)
    V, K = layout.n_views, nbr.shape[1]
    assert cam_from_world.dtype == torch.float64 and intr.dtype == torch.float64 and nbr.dtype == torch.int32
    assert tuple(cam_from_world.shape) == (V, 3, 4) and tuple(intr.shape) == (V, 4) and nbr.shape[0] == V
    pair = torch.empty((V, K, _lib.PAIR_TABLE_FLOATS), dtype=torch.float32, device=dev)
    src = torch.empty((V, 16), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_build_pair_tables_ragged(V, K, _p(layout.device(dev)), layout.host_ptr(), _p(cam_from_world), _p(intr),
                                                    _p(nbr), _p(pair), _p(src), _stream()))
    return pair, src


def backproject_filter_ragged(layout: ViewLayout, refined_all, normal, pair_table, src_table, vote_threshold: int,
                              opts: FilterOptions, bbox=None, xyz_out=None, votes_out=None, mark=None, support=None,
                              support_out=None):
    """Stages 2+3 for all views of ``layout``: refined_all flat [P] f32, normal flat [P,3] f32 (device, or pinned host).
    Returns xyz [G,3] f32 and votes [G] u8 on the views' strided grids (G = layout.total_grid); ``opts.stride`` must be
    the layout's stride.  ``support``, ``support_out``: as in ``backproject_filter`` (then also returns support [G] u8)."""
    lib = _lib.load()
    dev = _require_cuda_normal(normal, refined_all, pair_table, src_table, bbox, xyz_out, votes_out)
    V, P, G = layout.n_views, layout.total_pixels, layout.total_grid
    K = pair_table.shape[1]
    assert refined_all.dtype == torch.float32 and tuple(refined_all.shape) == (P,)
    assert normal.dtype == torch.float32 and tuple(normal.shape) == (P, 3)
    assert tuple(pair_table.shape) == (V, K, _lib.PAIR_TABLE_FLOATS) and tuple(src_table.shape) == (V, 16)
    if int(opts.stride) != layout.stride:
        raise ValueError(f"filter stride {opts.stride} but the layout was built for stride {layout.stride}")
    xyz = xyz_out if xyz_out is not None else torch.empty((G, 3), dtype=torch.float32, device=dev)
    votes = votes_out if votes_out is not None else torch.empty(G, dtype=torch.uint8, device=dev)
    cfg = opts.to_c()
    if support is not None:
        m, tau, rho = _support_args(support)
        sup = support_out if support_out is not None else torch.empty(G, dtype=torch.uint8, device=dev)
        assert sup.dtype == torch.uint8 and sup.is_contiguous() and tuple(sup.shape) == tuple(votes.shape)
        head = (C.byref(cfg), V, K, _p(layout.device(dev)), layout.host_ptr(), _p(refined_all), _p(normal),
                _p(pair_table), _p(src_table), int(vote_threshold), m, tau)
        tail = (_p(xyz), _p(votes), _p(sup), _p(bbox), C.byref(mark.c) if mark is not None else None, _stream())
        with torch.cuda.device(dev):
            if rho is None:
                _lib.check(lib.ddn_backproject_filter_support_ragged(*head, *tail))
            else:
                _lib.check(lib.ddn_backproject_filter_support_reproj_ragged(*head, rho, *tail))
        return xyz, votes, sup
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_backproject_filter_ragged(
                C.byref(cfg), V, K, _p(layout.device(dev)), layout.host_ptr(), _p(refined_all), _p(normal), _p(pair_table),
                _p(src_table), int(vote_threshold), _p(xyz), _p(votes), _p(bbox), C.byref(mark.c) if mark is not None else None,
                _stream(),
            )
        )
    return xyz, votes


def make_grid(bbox_min, bbox_max, voxel: float):
    """Voxel grid from a bounding box: origin = floor(min/voxel)*voxel in float32 (SURVEY.md N4) and the
    number of significant bits per axis."""
    v = np.float32(voxel)
    lo = np.asarray(bbox_min, dtype=np.float32)
    hi = np.asarray(bbox_max, dtype=np.float32)
    origin = (np.floor(lo / v) * v).astype(np.float32)
    cells = np.floor((hi - origin) / v).astype(np.int64) + 2
    bits = [max(1, int(math.ceil(math.log2(max(int(c), 2))))) for c in cells]
    if max(bits) > 21:
        raise DDNError(f"voxel grid needs {bits} bits per axis; the 3x21-bit key allows at most 21")
    g = _lib.VoxelGrid()
    g.voxel = float(v)
    for i in range(3):
        g.origin[i] = float(origin[i])
        g.bits[i] = bits[i]
        g.dims[i] = int(cells[i])
    return g


def checked_voxel_count(counts: torch.Tensor) -> int:
    """Number of voxels from the device counts [2] (synchronises); raises on the colour-sum overflow flag."""
    n_pts, mv = (int(x) for x in counts.cpu().tolist())
    if n_pts < 0:
        raise DDNError("voxel fusion: a voxel collected 2^24 or more points (32-bit colour sums); use a smaller voxel")
    return mv


GRID_STATUS = {0: "ok", 1: "empty (no finite bounding box)", 2: "grid larger than the session's capacity",
               3: "an axis needs more than 21 bits", 4: "fused through the hash table"}


class FuseSession:
    """Device buffers of one fusion session (include/ddn_b200.h: ddn_fuse_session): the grid lives on the device,
    derived there from bounding boxes, so a step runs without the host looking at an intermediate result.
    ``alloc(name, nbytes)`` may supply a buffer from elsewhere (NVLink-visible symmetric memory for ``units`` and
    ``tile_prefix`` in the multi-GPU path); every buffer is otherwise a plain device tensor."""

    def __init__(self, device, max_cells: int = 1 << 33, tile_prefix: bool = False, dirty: bool = True, alloc=None):
        lib = _lib.load()
        if not torch.cuda.is_available():
            raise DDNError("no CUDA device available: depthdensifier_b200 has no CPU fallback")
        self.device = torch.device(device)
        sizes = [C.c_int64(0) for _ in range(5)]
        _lib.check(lib.ddn_fuse_session_sizes(int(max_cells), *[C.byref(x) for x in sizes]))
        cap_units, units_b, dirty_b, sums_b, prefix_b = (x.value for x in sizes)
        self.max_cells, self.cap_units = int(max_cells), cap_units
        self.n_own_cap = cap_units // 256 + 2

        def get(name, nbytes):
            t = alloc(name, nbytes) if alloc is not None else None
            if t is None:
                t = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            assert t.is_cuda and t.is_contiguous() and t.numel() * t.element_size() >= nbytes and t.data_ptr() % 16 == 0
            return t

        self.units = get("units", units_b)
        self.dirty = get("dirty", dirty_b) if dirty else None
        self.tile_sums = get("tile_sums", sums_b)
        self.tile_prefix = get("tile_prefix", prefix_b) if tile_prefix else None
        self.grid = torch.zeros(16, dtype=torch.int32, device=self.device)
        self.counts = torch.zeros(2, dtype=torch.int64, device=self.device)
        self.c = _lib.FuseSession(self.grid.data_ptr(), self.units.data_ptr(), cap_units,
                                  self.dirty.data_ptr() if self.dirty is not None else None, self.tile_sums.data_ptr(),
                                  self.tile_prefix.data_ptr() if self.tile_prefix is not None else None, self.counts.data_ptr())
        self._accum = None
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_fuse_session_reset(C.byref(self.c), _stream()))

    def begin(self, boxes, voxel: float) -> None:
        """Opens a step on the union of ``boxes``: device tensors [6] (new_bbox encoding) or raw device addresses
        (peer memory)."""
        lib = _lib.load()
        ptrs = [b if isinstance(b, int) else b.data_ptr() for b in boxes]
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_fuse_begin(C.byref(self.c), arr, len(ptrs), float(np.float32(voxel)), _stream()))

    def begin_grid(self, grid: _lib.VoxelGrid) -> None:
        lib = _lib.load()
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_fuse_begin_grid(C.byref(self.c), C.byref(grid), _stream()))

    def grid_state(self) -> _lib.GridState:
        """Host copy of the device grid (synchronises)."""
        raw = self.grid.cpu().numpy().tobytes()
        return _lib.GridState.from_buffer_copy(raw)

    def host_grid(self) -> _lib.VoxelGrid:
        """The device grid as the host struct the host-grid entry points and the tests take (synchronises);
        raises when the session could not build one."""
        st = self.grid_state()
        if st.status == _lib.GRID_TOO_MANY_BITS:
            raise DDNError(f"fusion grid: {GRID_STATUS[st.status]} (dims {list(st.dims)}): the 3x21-bit voxel key cannot "
                           "address the bounding box at this voxel size; use a larger voxel")
        if st.status not in (_lib.GRID_OK, _lib.GRID_HASHED):
            raise DDNError(f"fusion grid: {GRID_STATUS.get(st.status, st.status)} (dims {list(st.dims)}, "
                           f"capacity {self.max_cells} cells); raise max_grid_cells or use a larger voxel")
        g = _lib.VoxelGrid()
        g.voxel = st.voxel
        for i in range(3):
            g.origin[i], g.bits[i], g.dims[i] = st.origin[i], st.bits[i], st.dims[i]
        return g

    def merge_scratch(self, world: int, cap_out: int) -> torch.Tensor:
        """Scratch of fuse_merge_peers for ``world`` ranks and ``cap_out`` records (allocated once per session)."""
        if getattr(self, "_merge_scratch", None) is None or self._merge_scratch[0] != (world, cap_out):
            nbytes = C.c_int64(0)
            _lib.check(_lib.load().ddn_fuse_merge_scratch_bytes(self.cap_units, int(world), int(cap_out), C.byref(nbytes)))
            self._merge_scratch = ((world, cap_out), torch.empty(nbytes.value, dtype=torch.uint8, device=self.device))
        return self._merge_scratch[1]

    def accum(self, cap_out: int) -> torch.Tensor:
        nbytes = cap_out * 40 + 16
        if self._accum is None or self._accum.numel() < nbytes:
            self._accum = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return self._accum

    def mark_points(self, xyz, votes, vote_threshold: int) -> None:
        lib = _lib.load()
        _require_cuda(xyz, votes)
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_fuse_mark_points(C.byref(self.c), xyz.shape[0], _p(xyz), _p(votes), int(vote_threshold), _stream()))


    def unmark_points(self, xyz) -> None:
        """N5: the cells of these points (xyz [N,3] f32, e.g. the sparse cloud) leave the occupancy, so no dense
        voxel is created there.  Between the mark and fuse_finish*."""
        lib = _lib.load()
        _require_cuda(xyz)
        assert xyz.dtype == torch.float32 and xyz.dim() == 2 and xyz.shape[1] == 3
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_fuse_unmark_points(C.byref(self.c), xyz.shape[0], _p(xyz), _stream()))


class HashFuse:
    """Buffers of the hashed fusion path (include/ddn_b200.h: struct ddn_hash_fuse) for steps of up to ``cap_voxels``
    points + dedup points: a table of 2x the next power of two >= cap_voxels slots (12 bytes each, at least 64 slots),
    the slot list and the sort buffers (28 bytes per point).  Allocated once and emptied; every step leaves the table empty again."""

    def __init__(self, device, cap_voxels: int):
        lib = _lib.load()
        if not torch.cuda.is_available():
            raise DDNError("no CUDA device available: depthdensifier_b200 has no CPU fallback")
        self.device = torch.device(device)
        self.cap_voxels = max(int(cap_voxels), 1)
        sizes = [C.c_int64(0) for _ in range(5)]
        _lib.check(lib.ddn_hash_fuse_sizes(self.cap_voxels, *[C.byref(x) for x in sizes]))
        self.cap_slots, table_b, slots_b, sort_b, hist_b = (x.value for x in sizes)
        new = lambda n: torch.empty(n, dtype=torch.uint8, device=self.device)
        self.table, self.slots, self.sort, self.hist = new(table_b), new(slots_b), new(sort_b), new(hist_b)
        self.state = torch.zeros(_lib.HASH_STATE_BYTES // 8, dtype=torch.int64, device=self.device)
        self.c = _lib.HashFuse(self.table.data_ptr(), self.slots.data_ptr(), self.sort.data_ptr(), self.hist.data_ptr(),
                               self.state.data_ptr(), self.cap_slots, self.cap_voxels)
        with torch.cuda.device(self.device):
            _lib.check(lib.ddn_hash_fuse_reset(C.byref(self.c), _stream()))

    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.table, self.slots, self.sort, self.hist, self.state))

    def ran(self) -> bool:
        """Whether the last step went through the hash table (synchronises)."""
        return int(self.state[0]) == 1

    def check(self) -> None:
        """Raises if the last step overflowed the table (synchronises); with ddn_hash_fuse_sizes' sizing it cannot."""
        check_hash_state(self.state[:2].tolist())

    def merge_scratch(self, world: int, cap_out: int) -> torch.Tensor:
        """Scratch of fuse_merge_hashed_peers for ``world`` ranks and ``cap_out`` records (allocated once)."""
        if getattr(self, "_merge_scratch", None) is None or self._merge_scratch[0] != (world, cap_out):
            nbytes = C.c_int64(0)
            _lib.check(_lib.load().ddn_fuse_merge_hashed_scratch_bytes(int(world), int(cap_out), C.byref(nbytes)))
            self._merge_scratch = None
            self._merge_scratch = ((world, cap_out), torch.empty(nbytes.value, dtype=torch.uint8, device=self.device))
        return self._merge_scratch[1]


def check_hash_state(state) -> None:
    """Raises on a host copy of the hash state words [ran, overflow] that report an incomplete step."""
    if int(state[0]) == 1 and int(state[1]) != 0:
        raise DDNError("hashed voxel fusion: table overflow, the step's voxels are incomplete")


def hashed_merge_capacity(n_max: int, world: int) -> int:
    """Records an owner of the hashed multi-GPU merge can receive when no rank has more than ``n_max`` points: at most
    n_max + ceil(2 world n_max / S) + 2 world (S = DDN_HASH_SAMPLES, DESIGN.md §6)."""
    return int(n_max) + -(-2 * int(world) * int(n_max) // _lib.HASH_SAMPLES) + 2 * int(world)


def new_hash_samples(dev) -> torch.Tensor:
    """Sample array of fuse_finish_hashed_partial: [DDN_HASH_SAMPLES + 1] i64."""
    return torch.empty(_lib.HASH_SAMPLES + 1, dtype=torch.int64, device=dev)


def new_voxel_outputs(cap_out: int, dev):
    return (torch.empty(cap_out, dtype=torch.int64, device=dev), torch.empty((cap_out, 3), dtype=torch.float32, device=dev),
            torch.empty((cap_out, 3), dtype=torch.uint8, device=dev), torch.empty(cap_out, dtype=torch.int32, device=dev))


def fuse_finish(sess: FuseSession, xyz, rgb, votes, vote_threshold: int, row_len: int = 0, cap_out: int | None = None, out=None):
    """Rank + accumulate + finalise of the points marked in ``sess``.  Returns keys, xyz, rgb, count (capacity
    ``cap_out``, default = the number of points) and the session's device counts [2] = (points, voxels)."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes)
    N = xyz.shape[0]
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and tuple(rgb.shape) == (N, 3)
    cap = max(int(cap_out if cap_out is not None else N), 1)
    k, x, c, n = out if out is not None else new_voxel_outputs(cap, dev)
    acc = sess.accum(cap)
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_finish(C.byref(sess.c), N, int(row_len), _p(xyz), _p(rgb), _p(votes), int(vote_threshold), _p(k), _p(x),
                                       _p(c), _p(n), cap, _p(acc), acc.numel(), _stream()))
    return k, x, c, n, sess.counts


def fuse_finish_hashed(sess: FuseSession, hf: HashFuse, xyz, rgb, votes, vote_threshold: int, row_len: int = 0,
                       dedup_xyz=None, mode: int = 0, cap_out: int | None = None, out=None):
    """Hashed fusion of the step's points (include/ddn_b200.h: ddn_fuse_finish_hashed).  ``mode`` 0: only when the
    session's grid is too large for its bitmap (the dense finish returns at once then); 1: on any grid.  ``dedup_xyz``
    [n,3] f32: N5, no voxel in the cells of these points.  Returns keys, xyz, rgb, count and the device counts [2], as
    fuse_finish; pass the same ``out`` as the dense finish so that one set of outputs holds whichever path ran."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes, dedup_xyz)
    N = xyz.shape[0]
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and tuple(rgb.shape) == (N, 3)
    assert dedup_xyz is None or (dedup_xyz.dtype == torch.float32 and dedup_xyz.dim() == 2 and dedup_xyz.shape[1] == 3)
    cap = max(int(cap_out if cap_out is not None else N), 1)
    k, x, c, n = out if out is not None else new_voxel_outputs(cap, dev)
    acc = sess.accum(max(cap, N))  # a voxel's accumulator is indexed by the point that created it
    n_dedup = 0 if dedup_xyz is None else dedup_xyz.shape[0]
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_finish_hashed(C.byref(sess.c), C.byref(hf.c), int(mode), N, int(row_len), _p(xyz), _p(rgb), _p(votes),
                                              int(vote_threshold), _p(dedup_xyz), n_dedup, _p(k), _p(x), _p(c), _p(n), cap, _p(acc),
                                              acc.numel(), _stream()))
    return k, x, c, n, sess.counts


def fuse_finish_hashed_partial(sess: FuseSession, hf: HashFuse, xyz, rgb, votes, vote_threshold: int, records, samples, row_len: int = 0,
                               dedup_xyz=None, mode: int = 0):
    """Hashed fusion of this rank's points into sorted partial ``records`` [cap, 6] i64 and ``samples``
    [DDN_HASH_SAMPLES + 1] i64 (include/ddn_b200.h: ddn_fuse_finish_hashed_partial); ``mode`` and ``dedup_xyz`` as
    fuse_finish_hashed.  Returns the session's device counts [2] = (points of this rank, records)."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes, records, samples, dedup_xyz)
    N = xyz.shape[0]
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and tuple(rgb.shape) == (N, 3)
    assert records.dtype == torch.int64 and records.shape[1] == _lib.RECORD_WORDS and records.is_contiguous()
    assert samples.dtype == torch.int64 and samples.numel() >= _lib.HASH_SAMPLES + 1
    assert dedup_xyz is None or (dedup_xyz.dtype == torch.float32 and dedup_xyz.dim() == 2 and dedup_xyz.shape[1] == 3)
    acc = sess.accum(max(N, 1))
    n_dedup = 0 if dedup_xyz is None else dedup_xyz.shape[0]
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_finish_hashed_partial(C.byref(sess.c), C.byref(hf.c), int(mode), N, int(row_len), _p(xyz), _p(rgb), _p(votes),
                                                      int(vote_threshold), _p(dedup_xyz), n_dedup, _p(records), records.shape[0],
                                                      _p(samples), _p(acc), acc.numel(), _stream()))
    return sess.counts


def fuse_merge_hashed_peers(sess: FuseSession, hf: HashFuse, rank: int, world: int, peer_records, peer_samples, plan, cap_out: int,
                            out=None):
    """Owner-side merge of the hashed partials over peer memory (include/ddn_b200.h: ddn_fuse_merge_hashed_peers); runs
    when this rank's fuse_finish_hashed_partial ran.  ``peer_*``: per rank, the device address of that rank's records /
    samples as mapped into this process.  ``cap_out`` (<= hf.cap_voxels): hashed_merge_capacity of the largest rank.
    Returns keys, xyz, rgb, count and the device counts, as fuse_merge_peers."""
    lib = _lib.load()
    dev = sess.device
    k, x, c, n = out if out is not None else new_voxel_outputs(cap_out, dev)
    scratch = hf.merge_scratch(world, cap_out)
    arr = lambda ptrs: (C.c_void_p * world)(*[int(v) for v in ptrs])
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_merge_hashed_peers(C.byref(sess.c), C.byref(hf.c), int(rank), int(world), arr(peer_records),
                                                   arr(peer_samples), _p(plan), _p(scratch), scratch.numel(), _p(k), _p(x), _p(c), _p(n),
                                                   int(cap_out), _stream()))
    return k, x, c, n, sess.counts


def fuse_finish_partial(sess: FuseSession, xyz, rgb, votes, vote_threshold: int, records, row_len: int = 0):
    """Rank + accumulate into partial ``records`` [cap, 6] i64 (and the session's tile prefix)."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes, records)
    N = xyz.shape[0]
    assert records.dtype == torch.int64 and records.shape[1] == _lib.RECORD_WORDS
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_finish_partial(C.byref(sess.c), N, int(row_len), _p(xyz), _p(rgb), _p(votes), int(vote_threshold),
                                               _p(records), records.shape[0], _stream()))
    return sess.counts


def fuse_merge_peers(sess: FuseSession, rank: int, world: int, peer_records, peer_tile_prefix, plan, cap_out: int, out=None,
                     drop_xyz=None):
    """Owner-side exchange + merge over peer memory.  ``peer_*``: per rank, the device address of that rank's
    records / tile prefix as mapped into this process.  ``drop_xyz`` [n,3] f32: N5, the sparse points of
    ALL ranks whose cells are removed from the merged occupancy.  Returns keys, xyz, rgb, count, counts."""
    lib = _lib.load()
    dev = sess.device
    k, x, c, n = out if out is not None else new_voxel_outputs(cap_out, dev)
    acc = sess.accum(cap_out)
    scratch = sess.merge_scratch(world, cap_out)
    arr = lambda ptrs: (C.c_void_p * world)(*[int(v) for v in ptrs])
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_fuse_merge_peers(C.byref(sess.c), int(rank), int(world), arr(peer_records), arr(peer_tile_prefix),
                                            _p(plan), _p(scratch), scratch.numel(), _p(drop_xyz),
                                            0 if drop_xyz is None else drop_xyz.shape[0], _p(k), _p(x), _p(c), _p(n), int(cap_out),
                                            _p(acc), acc.numel(), _stream()))
    return k, x, c, n, sess.counts


def voxel_fuse(xyz, rgb, votes, vote_threshold: int, grid: _lib.VoxelGrid, trim: bool = True, row_len: int = 0):
    """Stage 4.  xyz [N,3] f32, rgb [N,3] u8, votes [N] u8 or None.  Returns keys, xyz, rgb, count
    (trimmed to the voxel count when ``trim``; that reads the counts back and synchronises) and the
    device counts tensor [2] = (participating points, voxels).  ``row_len``: image width when the points
    are the pixels of row-major depth maps (locality hint only)."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes)
    N = xyz.shape[0]
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and tuple(rgb.shape) == (N, 3)
    assert votes is None or (votes.dtype == torch.uint8 and votes.numel() == N)
    nbytes = C.c_int64(0)
    _lib.check(lib.ddn_fuse_workspace_bytes(C.byref(grid), N, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    out_keys = torch.empty(N, dtype=torch.int64, device=dev)
    out_xyz = torch.empty((N, 3), dtype=torch.float32, device=dev)
    out_rgb = torch.empty((N, 3), dtype=torch.uint8, device=dev)
    out_cnt = torch.empty(N, dtype=torch.int32, device=dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_voxel_fuse(
                C.byref(grid), N, int(row_len), _p(xyz), _p(rgb), _p(votes), int(vote_threshold), _p(out_keys), _p(out_xyz),
                _p(out_rgb), _p(out_cnt), _p(counts), _p(ws), nbytes.value, _stream(),
            )
        )
    if trim:
        mv = checked_voxel_count(counts)
        return out_keys[:mv], out_xyz[:mv], out_rgb[:mv], out_cnt[:mv], counts
    return out_keys, out_xyz, out_rgb, out_cnt, counts


def fuse_tile_info(grid: _lib.VoxelGrid) -> tuple[int, int]:
    """(number of ownership tiles, cells per tile); 0 tiles = grid too large for the dense path."""
    lib = _lib.load()
    nt, cpt = C.c_int64(0), C.c_int64(0)
    _lib.check(lib.ddn_fuse_tile_info(C.byref(grid), C.byref(nt), C.byref(cpt)))
    return nt.value, cpt.value


def voxel_fuse_partial(xyz, rgb, votes, vote_threshold: int, grid: _lib.VoxelGrid, row_len: int = 0, tile_prefix=None,
                       out=None):
    """Rank-local stage 4: per-voxel partial RECORDS, keys ascending (layout: include/ddn_b200.h,
    ``unpack_records`` below).  Returns records [N, 6] i64 (sized for the worst case N) and the device
    counts [2] = (participating points, local voxels).  ``tile_prefix``: optional int32 [n_tiles + 1] output,
    the index of each tile's first record."""
    lib = _lib.load()
    dev = _require_cuda(xyz, rgb, votes)
    N = xyz.shape[0]
    assert xyz.dtype == torch.float32 and rgb.dtype == torch.uint8 and tuple(rgb.shape) == (N, 3)
    nbytes = C.c_int64(0)
    _lib.check(lib.ddn_fuse_workspace_bytes(C.byref(grid), N, C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    if out is not None:  # caller-provided record buffer (e.g. NVLink-visible symmetric memory)
        assert out.dtype == torch.int64 and out.is_contiguous() and out.shape[0] >= N and out.shape[1] == _lib.RECORD_WORDS
        rec = out
    else:
        rec = torch.empty((max(N, 1), _lib.RECORD_WORDS), dtype=torch.int64, device=dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_voxel_partials(
                C.byref(grid), N, int(row_len), _p(xyz), _p(rgb), _p(votes), int(vote_threshold), _p(rec), _p(tile_prefix),
                _p(counts), _p(ws), nbytes.value, _stream(),
            )
        )
    return rec, counts


def unpack_records(rec):
    """(keys, sums [n,3], colour sums [n,3], count) from records [n, 6] i64 (torch or numpy)."""
    lo = 0xFFFFFFFF
    return rec[:, 0], rec[:, 1:4], (rec[:, 4] >> 32) & lo, rec[:, 4] & lo, (rec[:, 5] >> 32) & lo, rec[:, 5] & lo


def voxel_merge_partials(records, grid: _lib.VoxelGrid, trim: bool = False, tile_range: tuple[int, int] = (0, 0)):
    """Owner-side merge of partial records [n, 6] i64 (any order) into final voxels.  ``tile_range``: the
    tiles this rank owns ((0, 0) = all); records of other tiles are ignored."""
    lib = _lib.load()
    dev = _require_cuda(records)
    n = records.shape[0]
    assert records.dtype == torch.int64 and (n == 0 or tuple(records.shape) == (n, _lib.RECORD_WORDS))
    nbytes = C.c_int64(0)
    _lib.check(lib.ddn_fuse_workspace_bytes(C.byref(grid), max(n, 1), C.byref(nbytes)))
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
    m = max(n, 1)
    out_keys = torch.empty(m, dtype=torch.int64, device=dev)
    out_xyz = torch.empty((m, 3), dtype=torch.float32, device=dev)
    out_rgb = torch.empty((m, 3), dtype=torch.uint8, device=dev)
    out_cnt = torch.empty(m, dtype=torch.int32, device=dev)
    counts = torch.zeros(2, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(
            lib.ddn_voxel_merge(
                C.byref(grid), n, _p(records), int(tile_range[0]), int(tile_range[1]), _p(out_keys), _p(out_xyz), _p(out_rgb),
                _p(out_cnt), _p(counts), _p(ws), nbytes.value, _stream(),
            )
        )
    if trim:
        mv = checked_voxel_count(counts)
        return out_keys[:mv], out_xyz[:mv], out_rgb[:mv], out_cnt[:mv], counts
    return out_keys, out_xyz, out_rgb, out_cnt, counts


def voxel_keys(xyz, voxel: float, origin) -> torch.Tensor:
    """Canonical 3x21-bit keys (int64 view of the uint64 key) for xyz [N,3] f32."""
    lib = _lib.load()
    dev = _require_cuda(xyz)
    g = _lib.VoxelGrid()
    g.voxel = float(np.float32(voxel))
    for i in range(3):
        g.origin[i] = float(np.float32(origin[i]))
        g.bits[i] = 21
        g.dims[i] = 0
    keys = torch.empty(xyz.shape[0], dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_voxel_keys(C.byref(g), xyz.shape[0], _p(xyz), _p(keys), _stream()))
    return keys


def project_points_device(points3d, cam_from_world34, kmat33):
    """float64 device form of the reference's project_points (scripts/test.py:58-76)."""
    lib = _lib.load()
    dev = _require_cuda(points3d, cam_from_world34, kmat33)
    n = points3d.shape[0]
    assert points3d.dtype == torch.float64 and cam_from_world34.dtype == torch.float64 and kmat33.dtype == torch.float64
    uv = torch.empty((n, 2), dtype=torch.float64, device=dev)
    z = torch.empty(n, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_project_points(n, _p(points3d), _p(cam_from_world34), _p(kmat33), _p(uv), _p(z), _stream()))
    return uv, z


def unproject_points_device(points2d, depth, params4):
    """float64 device form of the reference's unproject_points (scripts/test.py:79-90); depth is float32."""
    lib = _lib.load()
    dev = _require_cuda(points2d, depth)
    n = points2d.shape[0]
    assert points2d.dtype == torch.float64 and depth.dtype == torch.float32 and len(params4) == 4
    out = torch.empty((n, 3), dtype=torch.float64, device=dev)
    par = (C.c_double * 4)(*[float(v) for v in params4])
    with torch.cuda.device(dev):
        _lib.check(lib.ddn_unproject_points(n, _p(points2d), _p(depth), par, _p(out), _stream()))
    return out
