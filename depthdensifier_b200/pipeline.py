"""``main(ScriptConfig)``-compatible densification driver (reference: scripts/test.py:20-55, :58-90, :95-370).

Same configuration tree and tyro flags as the reference script (``--paths.recon-path``,
``--processing.downsample-density``, ``--filtering.vote-threshold`` ...), same stages, same output (a
COLMAP model with the kept dense points appended to the sparse ones), but

* the COLMAP model is read / written by ``colmap_io`` (the reference needs ``pycolmap``),
* all views are processed at once on the device by the batched kernels (align -> back-project + vote
  [-> voxel fusion]) instead of three Python loops; views of different sizes (several cameras, portrait and
  landscape shots) go through the ragged form of the same kernels, one flat pass over all views,
* MoGe inference is out of scope (BASELINE.json north_star): monocular depth / normal / mask come from a
  ``DepthProvider``.  ``PrecomputedDepth`` reads ``<depth_dir>/<image stem>.npz`` with arrays ``depth``
  [H,W] f32, ``normal`` [H,W,3] f32, ``mask`` [H,W] bool; ``MoGeDepth`` wraps the reference's model call
  (scripts/test.py:160-168) when the ``moge`` package and a checkpoint are present.

Reference-exact settings (the defaults): every view is tested against every processed view
(``filtering.num_neighbours = None``), nearest lookup, one-sided floater test, ``vote_threshold = 5``, no
voxel fusion (``fusion.voxel_size = None``: every kept point is appended).  The north-star settings are one
flag away: ``--filtering.num-neighbours 8 --fusion.voxel-size 0.01``.
"""

from __future__ import annotations

import dataclasses
import time
from dataclasses import dataclass, field
from pathlib import Path
from typing import Protocol

import numpy as np
import torch

from . import ops
from .colmap_io import Camera, Image, Reconstruction
from .ply import write_ply
from .depth_refiner import RefinerConfig
from .engine import DensifyConfig, DensifyEngine
from .neighbours import covisibility_table, nearest_views_table


# ==============================================================================================
# configuration (field for field scripts/test.py:20-55; additions are marked "new")
# ==============================================================================================
@dataclass
class PathsConfig:
    """Where the sparse model and the images are read from and where the densified model goes."""

    recon_path: Path = Path("data/360_v2/bicycle/sparse/0")
    image_dir: Path = Path("data/360_v2/bicycle/images")
    output_model_dir: Path = Path("results/0")
    depth_dir: Path | None = None
    """new: directory of precomputed <image stem>.npz (depth, normal, mask); None -> run MoGe."""
    output_ply: Path | None = None
    """new: also write the model's points as a binary PLY with oriented normals (x y z nx ny nz red green blue, the
    layout of COLMAP's fused.ply and 3DGS's points3D.ply): the sparse points with normal (0, 0, 0), then the dense
    points with their world-frame normals, turned toward the camera and fused per voxel with fusion.voxel_size."""


@dataclass
class MoGeConfig:
    """Monocular depth network (only used when no precomputed depth is given)."""

    checkpoint: Path = Path("models/moge/moge-2-vitl-normal/model.pt")


@dataclass
class ProcessingConfig:
    """Resolution and sampling density of the dense points."""

    pipeline_downsample_factor: int = 1
    """Images and cameras are shrunk by this integer factor before anything else (1 = full size)."""
    downsample_density: int = 32
    """Pixel stride of the back-projection grid: every n-th row and column yields a point."""


@dataclass
class FilteringConfig:
    """Multi-view consistency vote."""

    vote_threshold: int = 5
    """A point is dropped once this many views have voted against it (1..254)."""
    depth_threshold: float = 0.7
    """A view votes against a point that lies in front of the view's own surface by more than this ratio (z < T * D)."""
    num_neighbours: int | None = None
    """new: test each view against its K nearest views; None = against every view (reference)."""
    neighbour_mode: str = "covisibility"
    """new, with num_neighbours: 'covisibility' (views sharing the most sparse points) or 'nearest' (camera centres)."""
    sample_mode: str = "nearest"
    """new: 'nearest' (reference) or 'bilinear'."""
    min_support: int | None = None
    """new: also keep a point only when at least this many neighbour views see its surface within support_tau (relative
    depth error); None = no such test (reference), 0 = count only."""
    support_tau: float = 0.01
    """new, with min_support: the relative depth error |z - D| <= support_tau * D within which a view supports a point."""
    support_reproj_px: float | None = None
    """new, with min_support: a view supports a point only when, besides, the round trip source -> view -> source
    (forward-backward reprojection) lands within this many pixels of the point's pixel; None = no such test."""


@dataclass
class FusionConfig:
    """new: voxel-grid fusion of the kept points (the reference only concatenates).  Works for scenes of any extent:
    when the box of the back-projected points is too large for the dense occupancy bitmap (unbounded outdoor scenes,
    distant background, an outlier depth), the device fuses through a hash table sized by the points instead."""

    voxel_size: float | None = None
    dedup_sparse: bool = False
    """With voxel_size: no dense voxel is created where the sparse cloud already has a point (N5); the reference
    appends every dense point."""


@dataclass
class ScriptConfig:
    """Root of the configuration tree (same field names as the reference script, so the tyro flags match)."""

    paths: PathsConfig = field(default_factory=PathsConfig)
    moge: MoGeConfig = field(default_factory=MoGeConfig)
    processing: ProcessingConfig = field(default_factory=ProcessingConfig)
    refiner: RefinerConfig = field(default_factory=RefinerConfig)
    filtering: FilteringConfig = field(default_factory=FilteringConfig)
    fusion: FusionConfig = field(default_factory=FusionConfig)


# ==============================================================================================
# the reference's two helper functions, on the device
# ==============================================================================================
def project_points(points3d: np.ndarray, image: Image, camera: Camera) -> tuple[np.ndarray, np.ndarray]:
    """Projects 3D points to the image plane for a given camera (scripts/test.py:58-76): returns
    (points2d [N,2], depths [N]) in float64; no validity handling, the caller gates on depth > 0."""
    pts = torch.as_tensor(np.ascontiguousarray(points3d, dtype=np.float64).reshape(-1, 3)).cuda()
    pose = torch.as_tensor(np.ascontiguousarray(image.cam_from_world().matrix())).cuda()
    kmat = torch.as_tensor(np.ascontiguousarray(camera.calibration_matrix())).cuda()
    uv, z = ops.project_points_device(pts, pose, kmat)
    return uv.cpu().numpy(), z.cpu().numpy()


def unproject_points(points2D, depth, camera: Camera) -> np.ndarray:
    """Unprojects 2D image points to 3D camera coordinates (scripts/test.py:79-90); PINHOLE params."""
    fx, fy, cx, cy = camera.params
    uv = torch.as_tensor(np.ascontiguousarray(points2D, dtype=np.float64).reshape(-1, 2)).cuda()
    d = torch.as_tensor(np.ascontiguousarray(depth, dtype=np.float32).reshape(-1)).cuda()
    return ops.unproject_points_device(uv, d, (fx, fy, cx, cy)).cpu().numpy()


# ==============================================================================================
# monocular depth sources
# ==============================================================================================
class DepthProvider(Protocol):
    def __call__(self, image: Image, rgb: np.ndarray) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """rgb [H,W,3] u8 (already at processing resolution) -> depth [H,W] f32, normal [H,W,3] f32, mask [H,W] bool."""


class PrecomputedDepth:
    def __init__(self, depth_dir: Path):
        self.dir = Path(depth_dir)

    def __call__(self, image: Image, rgb: np.ndarray):
        path = self.dir / (Path(image.name).stem + ".npz")
        if not path.exists():
            raise FileNotFoundError(f"no precomputed depth for {image.name}: {path}")
        with np.load(path) as z:
            depth = np.asarray(z["depth"], dtype=np.float32)
            normal = np.asarray(z["normal"], dtype=np.float32) if "normal" in z.files else None
            mask = np.asarray(z["mask"], dtype=bool) if "mask" in z.files else depth > 0
        if normal is None:
            normal = np.zeros(depth.shape + (3,), np.float32)
            normal[..., 2] = -1.0
        if depth.shape != rgb.shape[:2]:
            raise ValueError(f"{path}: depth is {depth.shape}, the image at processing resolution is {rgb.shape[:2]}")
        return depth, normal, mask


class MoGeDepth:
    """The reference's model call (scripts/test.py:104-105, :153-168).  MoGe itself is third-party and out of
    scope; this wrapper exists so the driver is a drop-in when the package and weights are installed."""

    def __init__(self, checkpoint: Path, device):
        try:
            from moge.model.v2 import MoGeModel  # noqa: PLC0415
        except ImportError as e:  # pragma: no cover - moge is not in this image
            raise RuntimeError("the `moge` package is not installed: pass --paths.depth-dir with precomputed "
                               "<image>.npz depth / normal / mask maps instead") from e
        self.device = device
        self.model = MoGeModel.from_pretrained(checkpoint).to(device)
        self.model.eval()

    def __call__(self, image: Image, rgb: np.ndarray):  # pragma: no cover
        t = torch.from_numpy(rgb).permute(2, 0, 1).unsqueeze(0).float().div(255.0).to(self.device)
        with torch.no_grad():
            out = self.model.infer(t)
        return (out["depth"].squeeze(0).float().cpu().numpy(), out["normal"].squeeze(0).float().cpu().numpy(),
                out["mask"].squeeze(0).cpu().numpy().astype(bool))


def load_image_rgb(path: Path, factor: int) -> np.ndarray:
    """PIL open -> RGB -> LANCZOS resize by the integer factor (scripts/test.py:145-151)."""
    from PIL import Image as PILImage  # noqa: PLC0415

    im = PILImage.open(path).convert("RGB")
    w, h = im.size
    new_w, new_h = w // factor, h // factor
    if (new_w, new_h) != (w, h):
        im = im.resize((new_w, new_h), PILImage.Resampling.LANCZOS)
    return np.asarray(im)


# ==============================================================================================
# main
# ==============================================================================================
@dataclass
class DensifyOutput:
    reconstruction: Reconstruction
    points: np.ndarray  # [M,3] f64 appended points
    colors: np.ndarray  # [M,3] u8
    num_candidates: int  # valid pixels back-projected
    view_ids: list[int]
    timings: dict
    candidates: np.ndarray | None = None  # [N,3] f64 every back-projected point (return_candidates=True)
    keep: np.ndarray | None = None  # [N] bool
    normals: np.ndarray | None = None  # [M,3] f32 normals of the appended points (paths.output_ply)


def main(config: ScriptConfig, depth_provider: DepthProvider | None = None, return_candidates: bool = False) -> DensifyOutput:
    if not torch.cuda.is_available():
        raise ops.DDNError("depthdensifier_b200.pipeline.main needs a CUDA device: there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device())
    timings = {}
    t_total = time.time()

    # --- 1/2. depth source, COLMAP model ---
    t0 = time.time()
    if depth_provider is None:
        depth_provider = (PrecomputedDepth(config.paths.depth_dir) if config.paths.depth_dir is not None
                          else MoGeDepth(config.moge.checkpoint, dev))
    print(f"Loading COLMAP reconstruction from {config.paths.recon_path}...")
    rec = Reconstruction(config.paths.recon_path)
    print(f"Loaded model with {rec.num_reg_images()} images and {rec.num_points3D()} sparse points.")
    timings["load"] = time.time() - t0

    # --- 3/4a. gather the per-view inputs (host): sparse points, image, mono depth ---
    t0 = time.time()
    factor = max(int(config.processing.pipeline_downsample_factor), 1)
    views, depths, normals, masks, rgbs, sparse, poses, intr, observed = [], [], [], [], [], [], [], [], []
    for image in [im for im in rec.images.values() if im.has_pose]:
        pts = rec.sparse_xyz_of_image(image)
        if len(pts) == 0:  # scripts/test.py:136-137
            continue
        rgb = load_image_rgb(Path(config.paths.image_dir) / image.name, factor)
        new_h, new_w = rgb.shape[:2]
        depth, normal, mask = depth_provider(image, rgb)
        camera = rec.cameras[image.camera_id]
        camera.rescale(new_width=new_w, new_height=new_h)  # in place on the shared camera, as the reference does
        if camera.model_name != "PINHOLE":
            raise ValueError(f"camera {camera.camera_id} is {camera.model_name}; the reference's unproject_points "
                             "(scripts/test.py:81) only supports PINHOLE - undistort the model first")
        views.append(image.image_id)
        observed.append(image.observed_point3D_ids())
        depths.append(depth)
        normals.append(normal)
        masks.append(mask)
        rgbs.append(rgb)
        sparse.append(pts)
        poses.append(image.cam_from_world().matrix())
        intr.append(np.array(camera.params[:4], dtype=np.float64))
    if not views:
        raise ValueError("no registered image observes any sparse point")
    V = len(views)
    if (config.filtering.num_neighbours is None or config.filtering.num_neighbours >= V) and V > 1024:
        raise ValueError(f"{V} views: testing every view against every view (the reference's behaviour, K = V) is limited to "
                         "1024 views per call; set --filtering.num-neighbours (e.g. 8) to use a neighbour table")
    timings["inputs"] = time.time() - t0

    # --- 4b-6. device pipeline: align -> back-project + consistency vote [-> voxel fusion] ---
    t0 = time.time()
    K = config.filtering.num_neighbours
    poses_np = np.stack(poses)
    if K is None or K >= V:
        nbr = np.tile(np.arange(V, dtype=np.int32), (V, 1))  # every view incl. its own, in image order (reference)
    elif config.filtering.neighbour_mode == "covisibility":
        nbr = covisibility_table(observed, int(K), poses_np)
    elif config.filtering.neighbour_mode == "nearest":
        nbr = nearest_views_table(poses_np, int(K)).astype(np.int32)
    else:
        raise ValueError("filtering.neighbour_mode must be 'covisibility' or 'nearest'")
    rc = config.refiner
    align = ops.AlignOptions(min_correspondences=rc.min_correspondences, edge_margin=rc.edge_margin, robust=rc.robust,
                             outlier_threshold=rc.outlier_threshold, skip_smoothing=rc.skip_smoothing,
                             adaptive_correspondences=rc.adaptive_correspondences, zero_unmasked_passthrough=True)
    filt = ops.FilterOptions(depth_threshold=config.filtering.depth_threshold, sample_mode=config.filtering.sample_mode,
                             stride=max(int(config.processing.downsample_density), 1))
    ms, rp = config.filtering.min_support, config.filtering.support_reproj_px
    want_normals = config.paths.output_ply is not None
    eng = DensifyEngine(DensifyConfig(align=align, filter=filt, vote_threshold=int(config.filtering.vote_threshold),
                                      voxel=config.fusion.voxel_size, dedup_sparse=bool(config.fusion.dedup_sparse),
                                      min_support=None if ms is None else int(ms),
                                      support_tau=float(config.filtering.support_tau),
                                      support_reproj_px=None if rp is None else float(rp), fuse_normals=want_normals),
                        device=dev)
    offsets = np.concatenate([[0], np.cumsum([len(p) for p in sparse])]).astype(np.int64)
    to = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(dev)
    maps = ((depths, torch.float32), (normals, torch.float32), (masks, torch.bool), (rgbs, torch.uint8))
    if len({d.shape for d in depths}) == 1:
        run, maps = eng.run, [to(np.stack(m), dt) for m, dt in maps]
    else:  # views of different sizes: the ragged form of the device pipeline
        run, maps = eng.run_views, [[to(x, dt) for x in m] for m, dt in maps]
    res = run(*maps, to(poses_np, torch.float64), to(np.stack(intr), torch.float64), to(np.concatenate(sparse), torch.float64),
              to(offsets, torch.int64), to(nbr, torch.int32))
    n_candidates = res.num_points()
    nrm_out = None
    if config.fusion.voxel_size is None:
        pts, cols = res.kept_points()
        pts_out, col_out = pts.double().cpu().numpy(), cols.cpu().numpy()
        if want_normals:
            nrm_out = res.kept_normals().cpu().numpy()
    else:
        mv = int(res.counts[1].item()) if res.counts is not None else 0
        pts_out = res.voxel_xyz[:mv].double().cpu().numpy() if mv else np.zeros((0, 3))
        col_out = res.voxel_rgb[:mv].cpu().numpy() if mv else np.zeros((0, 3), np.uint8)
        if want_normals:
            nrm_out = res.voxel_normal[:mv].cpu().numpy() if mv else np.zeros((0, 3), np.float32)
    torch.cuda.synchronize(dev)
    timings["device_pipeline"] = time.time() - t0
    print(f"-> {n_candidates} candidate points from {V} views, {len(pts_out)} kept"
          + (f" ({config.fusion.voxel_size} voxels)" if config.fusion.voxel_size is not None else ""))

    # --- 7. merge with the sparse cloud and save (scripts/test.py:353-364) ---
    t0 = time.time()
    rec.add_points3D(pts_out, col_out)
    out_dir = Path(config.paths.output_model_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    rec.write_binary(out_dir)
    if want_normals:
        sparse_pts = [rec.points3D[pid] for pid in sorted(rec.points3D)]
        sp_xyz = np.array([p.xyz for p in sparse_pts], np.float64).reshape(-1, 3)
        sp_rgb = np.array([p.color for p in sparse_pts], np.uint8).reshape(-1, 3)
        Path(config.paths.output_ply).parent.mkdir(parents=True, exist_ok=True)
        write_ply(config.paths.output_ply, np.concatenate([sp_xyz, pts_out]), np.concatenate([np.zeros_like(sp_xyz), nrm_out]),
                  np.concatenate([sp_rgb, col_out]))
    timings["write"] = time.time() - t0
    timings["total"] = time.time() - t_total
    print(f"Saved model with {rec.num_points3D()} points to {out_dir} (total {timings['total']:.2f}s)")
    out = DensifyOutput(rec, pts_out, col_out, n_candidates, views, timings, normals=nrm_out)
    if return_candidates:
        valid = res.votes != 255
        out.candidates = res.xyz[valid].double().cpu().numpy()
        out.keep = (res.votes[valid] < res.fusion_threshold()).cpu().numpy()
    return out


def cli() -> None:
    import tyro  # noqa: PLC0415

    main(tyro.cli(ScriptConfig))


if __name__ == "__main__":
    cli()
