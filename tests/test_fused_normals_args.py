"""The fused-normal option's argument checks without a GPU: DensifyConfig, ShardedDensifier, the CLI flag and the C
entry points."""

import ctypes as C

import numpy as np
import pytest
import torch

from depthdensifier_b200.engine import DensifyConfig


def test_densify_config_default_off():
    assert DensifyConfig().fuse_normals is False
    assert DensifyConfig(fuse_normals=True).fuse_normals is True


def test_sharded_densifier_refuses_normals():
    from depthdensifier_b200.distributed import ShardedDensifier

    poses = torch.zeros((2, 3, 4), dtype=torch.float64)
    with pytest.raises(ValueError, match="multi-GPU form"):
        ShardedDensifier(DensifyConfig(fuse_normals=True), "cpu", 0, 1, 2, 0, 2, poses, torch.zeros((2, 4), dtype=torch.float64),
                         np.zeros((2, 1), np.int32), 8, 8, backend=object())


def test_cli_flag(tmp_path):
    tyro = pytest.importorskip("tyro")
    from depthdensifier_b200 import pipeline as P

    cfg = tyro.cli(P.ScriptConfig, args=["--paths.output-ply", str(tmp_path / "o.ply")])
    assert cfg.paths.output_ply == tmp_path / "o.ply"
    assert tyro.cli(P.ScriptConfig, args=[]).paths.output_ply is None


def test_entry_points_reject_bad_arguments(lib_built):
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    assert lib.ddn_point_normals(2, 8, 8, 0, None, None, None, None, None, None) != 0  # stride 0
    assert b"stride" in lib.ddn_last_error_string()
    assert lib.ddn_point_normals(2, 8, 8, 1, None, None, None, None, None, None) != 0  # null pointers
    assert lib.ddn_point_normals(0, 8, 8, 1, None, None, None, None, None, None) == 0  # no views: nothing to do
    assert lib.ddn_point_normals_ragged(1, None, None, None, None, None, None, None, None) != 0  # no host layout
    g = _lib.VoxelGrid()
    g.voxel = 0.1
    for i in range(3):
        g.bits[i], g.dims[i] = 8, 0
    plain, normals = C.c_int64(0), C.c_int64(0)
    assert lib.ddn_fuse_workspace_bytes(C.byref(g), 1000, C.byref(plain)) == 0
    assert lib.ddn_fuse_normals_workspace_bytes(C.byref(g), 1000, C.byref(normals)) == 0
    assert normals.value >= plain.value + 1000 * 24  # three more u64 per possible voxel
    assert lib.ddn_voxel_fuse_normals(C.byref(g), 10, 0, None, None, None, 1, None, None, None, None, None, None, None, None, 0,
                                      None) != 0
    sess = _lib.FuseSession()
    assert lib.ddn_fuse_finish_normals(C.byref(sess), 10, 0, None, None, None, 1, None, None, None, None, None, None, 16, None, 0,
                                       None) != 0
    hf = _lib.HashFuse()
    assert lib.ddn_fuse_finish_hashed_normals(C.byref(sess), C.byref(hf), 0, 10, 0, None, None, None, 1, None, None, 0, None, None,
                                              None, None, None, 16, None, 0, None) != 0
