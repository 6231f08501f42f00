"""ctypes binding of libddn_b200.so (the C ABI declared in include/ddn_b200.h).

There is no CPU fallback: if the library is missing, or no CUDA device is present when a compute
entry point is called, this module raises.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

PKG_DIR = Path(__file__).resolve().parent
# DDN_LIB_PATH: load another build of the same library (kernel tuning experiments: build.py --suffix)
LIB_PATH = Path(os.environ["DDN_LIB_PATH"]) if os.environ.get("DDN_LIB_PATH") else PKG_DIR / "libddn_b200.so"


class DDNError(RuntimeError):
    pass


class AlignConfig(C.Structure):
    _fields_ = [
        ("min_correspondences", C.c_int32),
        ("edge_margin", C.c_int32),
        ("robust", C.c_int32),
        ("outlier_threshold", C.c_float),
        ("skip_smoothing", C.c_int32),
        ("adaptive_correspondences", C.c_int32),
        ("max_pairs", C.c_int32),
        ("mode", C.c_int32),
        ("subsample_seed", C.c_uint32),
        ("zero_unmasked_passthrough", C.c_int32),
        ("mask_packed", C.c_int32),
        ("use_tma", C.c_int32),
    ]


class ViewStats(C.Structure):
    _fields_ = [
        ("status", C.c_int32),
        ("num_correspondences", C.c_int32),
        ("outliers_removed", C.c_int32),
        ("num_table", C.c_int32),
        ("scale_factor", C.c_float),
        ("affine_scale", C.c_float),
        ("affine_shift", C.c_float),
        ("reserved", C.c_int32),
    ]


class FilterConfig(C.Structure):
    _fields_ = [
        ("depth_threshold", C.c_float),
        ("grazing_cos", C.c_float),
        ("sample_mode", C.c_int32),
        ("two_sided_tau", C.c_float),
        ("stride", C.c_int32),
        ("normals_in_world", C.c_int32),
        ("pixel_layout", C.c_int32),
    ]


class VoxelGrid(C.Structure):
    _fields_ = [("voxel", C.c_float), ("origin", C.c_float * 3), ("bits", C.c_int32 * 3), ("dims", C.c_int32 * 3)]


class GridState(C.Structure):
    """ddn_grid_state: the device-resident grid of a fusion session (64 bytes)."""

    _fields_ = [("voxel", C.c_float), ("origin", C.c_float * 3), ("bits", C.c_int32 * 3), ("dims", C.c_int32 * 3),
                ("n_units", C.c_int64), ("status", C.c_int32), ("reserved", C.c_int32), ("cells", C.c_int64)]


class FuseSession(C.Structure):
    """ddn_fuse_session: host struct of device pointers."""

    _fields_ = [("grid", C.c_void_p), ("units", C.c_void_p), ("cap_units", C.c_int64), ("dirty", C.c_void_p),
                ("tile_sums", C.c_void_p), ("tile_prefix", C.c_void_p), ("counts", C.c_void_p)]


class HashFuse(C.Structure):
    """struct ddn_hash_fuse: host struct of device pointers (the hashed fusion path's buffers)."""

    _fields_ = [("table", C.c_void_p), ("slots", C.c_void_p), ("sort", C.c_void_p), ("hist", C.c_void_p), ("state", C.c_void_p),
                ("cap_slots", C.c_int64), ("cap_voxels", C.c_int64)]


GRID_OK, GRID_EMPTY, GRID_TOO_LARGE, GRID_TOO_MANY_BITS, GRID_HASHED = 0, 1, 2, 3, 4
HASH_STATE_BYTES = 64  # DDN_HASH_STATE_BYTES
MAX_PEERS = 16
PAIR_TABLE_FLOATS = 24
LAYOUT_COLS = 8  # DDN_LAYOUT_COLS
RECORD_WORDS = 6  # DDN_RECORD_WORDS
RECORD_NORMAL_WORDS = 10  # DDN_RECORD_NORMAL_WORDS: the partial records of the fused-normal forms
HASH_SAMPLES = 4096  # DDN_HASH_SAMPLES

# every symbol include/ddn_b200.h declares: name -> (restype, argtypes)
_vp, _i64, _i32 = C.c_void_p, C.c_int64, C.c_int32
SYMBOLS = {
    "ddn_version": (C.c_int, []),
    "ddn_last_error_string": (C.c_char_p, []),
    "ddn_launch_count": (C.c_int64, []),
    "ddn_debug_peer_read": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _vp]),
    "ddn_profile_enable": (None, [C.c_int]),
    "ddn_profile_report": (C.c_int, [C.c_char_p, C.c_int64]),
    "ddn_align_config_default": (None, [C.POINTER(AlignConfig)]),
    "ddn_filter_config_default": (None, [C.POINTER(FilterConfig)]),
    "ddn_align_workspace_bytes": (C.c_int, [_i64, _i64, C.POINTER(_i64)]),
    "ddn_align_views": (
        C.c_int,
        [C.POINTER(AlignConfig), _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp],
    ),
    "ddn_build_pair_tables": (C.c_int, [_i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ddn_backproject_filter": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp,
         C.POINTER(FuseSession), _vp],
    ),
    "ddn_backproject_filter_support": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32, C.c_float, _vp, _vp,
         _vp, _vp, C.POINTER(FuseSession), _vp],
    ),
    "ddn_backproject_filter_support_reproj": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _i32, C.c_float,
         C.c_float, _vp, _vp, _vp, _vp, C.POINTER(FuseSession), _vp],
    ),
    "ddn_bbox_init": (C.c_int, [_vp, _vp]),
    "ddn_align_views_ragged": (
        C.c_int,
        [C.POINTER(AlignConfig), _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp],
    ),
    "ddn_build_pair_tables_ragged": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ddn_backproject_filter_ragged": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, C.POINTER(FuseSession), _vp],
    ),
    "ddn_backproject_filter_support_ragged": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, C.c_float, _vp, _vp, _vp, _vp,
         C.POINTER(FuseSession), _vp],
    ),
    "ddn_backproject_filter_support_reproj_ragged": (
        C.c_int,
        [C.POINTER(FilterConfig), _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, C.c_float, C.c_float, _vp, _vp, _vp,
         _vp, C.POINTER(FuseSession), _vp],
    ),
    "ddn_pchip_workspace_bytes": (C.c_int, [_i64, _i64, C.POINTER(_i64)]),
    "ddn_pchip_edge_mask": (
        C.c_int,
        [_i64, _i64, _vp, _vp, _vp, _vp, C.POINTER(C.c_double), _i32, C.c_float, C.c_double, _vp, _vp, _i64, _vp],
    ),
    "ddn_pchip_apply": (C.c_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp]),
    "ddn_gradient_mask": (
        C.c_int,
        [_i64, _i64, _vp, _vp, C.POINTER(C.c_float), _i32, C.c_float, C.c_float, _vp, _vp, _i64, _vp],
    ),
    "ddn_transform_normals": (C.c_int, [_i64, _vp, C.POINTER(C.c_double), _i32, _vp, _vp]),
    "ddn_project_points": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ddn_unproject_points": (C.c_int, [_i64, _vp, _vp, C.POINTER(C.c_double), _vp, _vp]),
    "ddn_point_normals": (C.c_int, [_i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ddn_point_normals_ragged": (C.c_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ddn_fuse_workspace_bytes": (C.c_int, [C.POINTER(VoxelGrid), _i64, C.POINTER(_i64)]),
    "ddn_fuse_normals_workspace_bytes": (C.c_int, [C.POINTER(VoxelGrid), _i64, C.POINTER(_i64)]),
    "ddn_voxel_fuse_normals": (
        C.c_int,
        [C.POINTER(VoxelGrid), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    ),
    "ddn_voxel_fuse": (
        C.c_int,
        [C.POINTER(VoxelGrid), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    ),
    "ddn_fuse_tile_info": (C.c_int, [C.POINTER(VoxelGrid), C.POINTER(_i64), C.POINTER(_i64)]),
    "ddn_voxel_partials": (
        C.c_int,
        [C.POINTER(VoxelGrid), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp],
    ),
    "ddn_voxel_merge": (
        C.c_int,
        [C.POINTER(VoxelGrid), _i64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    ),
    "ddn_voxel_keys": (C.c_int, [C.POINTER(VoxelGrid), _i64, _vp, _vp, _vp]),
    "ddn_fuse_session_sizes": (C.c_int, [_i64] + [C.POINTER(_i64)] * 5),
    "ddn_fuse_merge_scratch_bytes": (C.c_int, [_i64, _i32, _i64, C.POINTER(_i64)]),
    "ddn_fuse_merge_normals_scratch_bytes": (C.c_int, [_i64, _i32, _i64, C.POINTER(_i64)]),
    "ddn_fuse_session_reset": (C.c_int, [C.POINTER(FuseSession), _vp]),
    "ddn_fuse_begin": (C.c_int, [C.POINTER(FuseSession), C.POINTER(_vp), _i32, C.c_float, _vp]),
    "ddn_fuse_begin_grid": (C.c_int, [C.POINTER(FuseSession), C.POINTER(VoxelGrid), _vp]),
    "ddn_fuse_mark_points": (C.c_int, [C.POINTER(FuseSession), _i64, _vp, _vp, _i32, _vp]),
    "ddn_fuse_unmark_points": (C.c_int, [C.POINTER(FuseSession), _i64, _vp, _vp]),
    "ddn_fuse_finish": (
        C.c_int,
        [C.POINTER(FuseSession), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_fuse_finish_normals": (
        C.c_int,
        [C.POINTER(FuseSession), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_fuse_finish_partial": (C.c_int, [C.POINTER(FuseSession), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _i64, _vp]),
    "ddn_fuse_finish_partial_normals": (C.c_int, [C.POINTER(FuseSession), _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp]),
    "ddn_fuse_merge_peers": (
        C.c_int,
        [C.POINTER(FuseSession), _i32, _i32, C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _i64, _vp, _i64,
         _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_fuse_merge_peers_normals": (
        C.c_int,
        [C.POINTER(FuseSession), _i32, _i32, C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _i64, _vp, _i64,
         _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_hash_fuse_sizes": (C.c_int, [_i64] + [C.POINTER(_i64)] * 5),
    "ddn_hash_fuse_reset": (C.c_int, [C.POINTER(HashFuse), _vp]),
    "ddn_fuse_finish_hashed": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _i64,
         _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_fuse_finish_hashed_normals": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _i64,
         _vp, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _vp],
    ),
    "ddn_fuse_finish_hashed_partial": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp],
    ),
    "ddn_fuse_finish_hashed_partial_normals": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _i64,
         _vp],
    ),
    "ddn_fuse_merge_hashed_scratch_bytes": (C.c_int, [_i32, _i64, C.POINTER(_i64)]),
    "ddn_fuse_merge_hashed_normals_scratch_bytes": (C.c_int, [_i32, _i64, C.POINTER(_i64)]),
    "ddn_fuse_merge_hashed_peers": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i32, C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _i64, _vp, _vp, _vp, _vp,
         _i64, _vp],
    ),
    "ddn_fuse_merge_hashed_peers_normals": (
        C.c_int,
        [C.POINTER(FuseSession), C.POINTER(HashFuse), _i32, _i32, C.POINTER(_vp), C.POINTER(_vp), _vp, _vp, _i64, _vp, _vp, _vp, _vp,
         _vp, _i64, _vp],
    ),
}

_lib = None


def load():
    """Load the shared library (once) and declare prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise DDNError(
            f"{LIB_PATH} is missing: build it with `python -m depthdensifier_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.ddn_version() != 200:
        raise DDNError(f"libddn_b200.so version mismatch: {lib.ddn_version()}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().ddn_last_error_string().decode("utf-8", "replace")
        raise DDNError(f"libddn_b200 error {rc}: {msg}")


def profile(on: bool) -> None:
    load().ddn_profile_enable(1 if on else 0)


def profile_report() -> list[tuple[str, float]]:
    """[(kernel, ms since the previous mark)] recorded since profile(True); synchronises."""
    buf = C.create_string_buffer(1 << 20)
    check(load().ddn_profile_report(buf, len(buf)))
    rows = [ln.rsplit(" ", 1) for ln in buf.value.decode().splitlines() if ln]
    return [(a, float(b)) for a, b in rows]


def launch_count() -> int:
    return int(load().ddn_launch_count())
