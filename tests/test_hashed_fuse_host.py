"""Host-side checks of the hashed fusion path: its C struct and sizes, the synthetic dome background, and that the dome
scene of tests/test_gpu_hashed_fuse.py really cannot be fused by the dense path."""

import ctypes
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from depthdensifier_b200.synthetic import SceneConfig, make_scene

ROOT = Path(__file__).resolve().parent.parent


def test_hash_fuse_struct_matches_the_header(tmp_path):
    """struct ddn_hash_fuse, compiled as C, has the size and field offsets of its ctypes mirror."""
    from depthdensifier_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    names = [n for n, *_ in _lib.HashFuse._fields_]
    lines = ["#include <stddef.h>", "#include <stdio.h>", f'#include "{ROOT / "include" / "ddn_b200.h"}"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(struct ddn_hash_fuse));']
    lines += [f'  printf("{n} %zu\\n", offsetof(struct ddn_hash_fuse, {n}));' for n in names]
    lines += [f'  printf("state_bytes %d\\n", DDN_HASH_STATE_BYTES);', f'  printf("hashed %d\\n", DDN_GRID_HASHED);', "  return 0;", "}"]
    src = tmp_path / "hash_layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "hash_layout"
    subprocess.run([gcc, "-std=c11", "-Wall", "-Werror", "-o", str(exe), str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(_lib.HashFuse)
    for n in names:
        assert int(got[n]) == getattr(_lib.HashFuse, n).offset, n
    assert int(got["state_bytes"]) == _lib.HASH_STATE_BYTES and int(got["hashed"]) == _lib.GRID_HASHED


def test_hash_fuse_sizes_and_argument_checks(lib_built):
    """The table has 2x the next power of two >= cap_voxels slots, at least 64 (at most half full); invalid calls fail
    before any launch."""
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    out = [ctypes.c_int64(0) for _ in range(5)]
    for cap, slots in [(1, 64), (31, 64), (1000, 2048), (1024, 2048), (1025, 4096)]:
        assert lib.ddn_hash_fuse_sizes(cap, *[ctypes.byref(x) for x in out]) == 0
        assert out[0].value == slots and out[1].value == 12 * slots and out[2].value >= 4 * cap and out[3].value >= 24 * cap
    assert lib.ddn_hash_fuse_sizes(0, *[ctypes.byref(x) for x in out]) == -1
    sess, hf = _lib.FuseSession(), _lib.HashFuse()
    assert lib.ddn_fuse_finish_hashed(ctypes.byref(sess), ctypes.byref(hf), 0, 10, 0, None, None, None, 1, None, 0, None, None, None,
                                      None, 10, None, 0, None) == -1
    assert b"invalid argument" in lib.ddn_last_error_string()


@pytest.mark.parametrize("large", [False, True], ids=["dense", "over_2e35_cells"])
def test_host_grid_workspace_is_checked_before_any_launch(lib_built, large):
    """ddn_fuse_workspace_bytes sizes ddn_voxel_fuse, ddn_voxel_partials and ddn_voxel_merge on a dense grid and on one of
    more than 2^35 cells (the hashed path, also the size for grid NULL); 16 bytes less makes each of them return
    DDN_ERR_WORKSPACE_TOO_SMALL without launching anything (the dummy device pointers are never touched)."""
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    g = _lib.VoxelGrid()
    g.voxel = 0.01
    for i, d in enumerate([4000, 4000, 4000] if large else [100, 80, 60]):
        g.bits[i] = int(d - 1).bit_length()
        g.dims[i] = d
    assert (int(g.dims[0]) * g.dims[1] * g.dims[2] > 2**35) == large
    n = 100_000
    nbytes = ctypes.c_int64(0)
    assert lib.ddn_fuse_workspace_bytes(ctypes.byref(g), n, ctypes.byref(nbytes)) == 0
    if large:
        assert 100 * n <= nbytes.value <= 124 * n + (1 << 17)
        null_bytes = ctypes.c_int64(0)
        assert lib.ddn_fuse_workspace_bytes(None, n, ctypes.byref(null_bytes)) == 0 and null_bytes.value == nbytes.value
    ws, short = ctypes.c_void_p(1 << 20), nbytes.value - 16
    p = ctypes.c_void_p(1 << 12)  # any 256-byte aligned address
    too_small = -3  # DDN_ERR_WORKSPACE_TOO_SMALL
    assert lib.ddn_voxel_fuse(ctypes.byref(g), n, 0, p, p, None, 1, p, p, p, p, p, ws, short, None) == too_small
    assert lib.ddn_voxel_partials(ctypes.byref(g), n, 0, p, p, None, 1, p, None, p, ws, short, None) == too_small
    assert lib.ddn_voxel_merge(ctypes.byref(g), n, p, 0, 0, p, p, p, p, p, ws, short, None) == too_small
    assert b"workspace too small" in lib.ddn_last_error_string()


def test_default_scene_is_unchanged(golden_dir):
    """dome_radius=None (the default) leaves every scene as it was: the seed-11 scene of the golden reference run."""
    g = np.load(golden_dir / "ref_main_seed11.npz")
    sc = make_scene(SceneConfig(n_views=5, width=112, height=80, n_sparse=600, seed=11, dome_radius=None))
    for k in ("mask", "rgb", "sparse_offsets"):
        assert np.array_equal(getattr(sc, k).numpy(), g[k]), k
    for k in ("mono_depth", "normal", "sparse_xyz", "cam_from_world", "intrinsics"):
        np.testing.assert_allclose(getattr(sc, k).numpy(), g[k], rtol=1e-6, atol=1e-7, err_msg=k)


def test_dome_scene_box_exceeds_the_dense_bitmap():
    """The dome scene the GPU tests fuse: every pixel sees something, and the box of the surface its views see holds more
    than 2^35 cells at the test voxel size (the most any dense session can hold), with every axis within 2^21 cells."""
    from test_gpu_hashed_fuse import DOME, DOME_VOXEL

    sc = make_scene(SceneConfig(**DOME))
    assert bool(sc.mask.all())
    V, H, W = sc.mono_depth.shape
    fx, fy, cx, cy = sc.intrinsics[0].tolist()
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing="ij")
    dir_cam = np.stack([(xs - cx) / fx, (ys - cy) / fy, np.ones((H, W))], -1)
    pts = []
    for v in range(V):
        Rm, t = sc.cam_from_world[v, :, :3].numpy(), sc.cam_from_world[v, :, 3].numpy()
        pts.append((-Rm.T @ t) + sc.true_depth[v].numpy()[..., None].astype(np.float64) * (dir_cam @ Rm))
    p = np.concatenate([x.reshape(-1, 3) for x in pts])
    cells = np.floor((p.max(0) - p.min(0)) / DOME_VOXEL) + 2
    assert np.prod(cells) > 4 * 2.0**35 and (cells < 2**21).all()
    # without the dome, the pixels that see nothing are masked out
    plain = make_scene(SceneConfig(**{**DOME, "dome_radius": None}))
    assert not bool(plain.mask.all())
