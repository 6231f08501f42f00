"""Views of different sizes without a GPU: the ragged layout (include/ddn_b200.h, DDN_LAYOUT_COLS), the host-side argument
checks of the ragged entry points, and the per-view list form of the oracle (tests/ragged_oracle.py)."""

import ctypes

import numpy as np
import pytest

from depthdensifier_b200.neighbours import nearest_views_table
from depthdensifier_b200.synthetic import SceneConfig, make_scene
from oracle import restatement as R

import ragged_oracle


def test_layout_offsets_and_prefixes():
    from depthdensifier_b200.ops import ViewLayout

    shapes = [(840, 1297), (1297, 840), (2, 5), (33, 127)]
    L = ViewLayout.from_shapes(shapes, stride=3)
    t = L.table
    assert t.dtype == np.int64 and t.shape == (5, 8)
    assert t[:4, :2].tolist() == [list(s) for s in shapes]
    pix = [h * w for h, w in shapes]
    grid = [((h + 2) // 3) * ((w + 2) // 3) for h, w in shapes]
    tiles = [((h + 31) // 32) * ((w + 125) // 126) for h, w in shapes]
    chunks = [(g + 1023) // 1024 for g in grid]
    for col, units in ((2, pix), (3, grid), (4, tiles), (5, chunks)):
        assert t[:, col].tolist() == np.concatenate([[0], np.cumsum(units)]).tolist()
    assert t[4, 0] == 3 and t[4, 1] == 4 and (t[:, 6:] == 0).all()
    assert L.total_pixels == sum(pix) and L.total_grid == sum(grid) and L.grid_shapes[2] == (1, 2)
    assert not L.uniform and ViewLayout.from_shapes([(4, 5)] * 3).uniform
    # split / flatten round trip on host tensors
    import torch

    maps = [torch.arange(h * w, dtype=torch.float32).view(h, w) + v for v, (h, w) in enumerate(shapes)]
    flat = L.flatten(maps)
    assert flat.shape == (sum(pix),)
    assert all(torch.equal(a, b) for a, b in zip(L.split(flat), maps))
    g = torch.arange(L.total_grid)
    assert [tuple(x.shape) for x in L.split(g, grid=True)] == L.grid_shapes


def test_layout_rejections():
    from depthdensifier_b200.ops import ViewLayout

    with pytest.raises(ValueError, match="2\\^32"):
        ViewLayout.from_shapes([(65535, 32768)] * 2 + [(256, 256)])  # 2^32 pixels
    assert ViewLayout.from_shapes([(65535, 32768)] * 2 + [(256, 255)]).total_pixels == (1 << 32) - 256
    with pytest.raises(ValueError, match="zero-sized"):
        ViewLayout.from_shapes([(4, 4), (0, 7)])
    with pytest.raises(ValueError, match="65535"):
        ViewLayout.from_shapes([(2, 2)] * 65536)
    with pytest.raises(ValueError):
        ViewLayout.from_shapes([])
    with pytest.raises(ValueError):
        ViewLayout.from_shapes([(1 << 22, 2)])


def test_ragged_entry_points_validate_without_gpu(lib_built):
    """Host-side checks only: every call below fails before any kernel or CUDA call."""
    from depthdensifier_b200 import _lib
    from depthdensifier_b200.ops import ViewLayout

    lib = _lib.load()
    L = ViewLayout.from_shapes([(40, 60), (61, 33)], stride=2)
    host = L.host_ptr()
    fake = ctypes.c_void_p(0x10000)  # never dereferenced: validation fails first
    acfg = _lib.AlignConfig()
    lib.ddn_align_config_default(ctypes.byref(acfg))

    def align(cfg, layout, layout_host):
        return lib.ddn_align_views_ragged(ctypes.byref(cfg), 2, layout, layout_host, fake, None, fake, fake, fake, fake, 10, fake,
                                          fake, fake, 1 << 20, None, None, None)

    assert align(acfg, None, host) == -1 and b"null layout" in lib.ddn_last_error_string()
    acfg.use_tma = 1
    assert align(acfg, fake, host) == -4 and b"use_tma" in lib.ddn_last_error_string()
    acfg.use_tma, acfg.mask_packed = 0, 1
    assert align(acfg, fake, host) == -4
    acfg.mask_packed = 0
    assert align(acfg, fake, None) == -1
    bad = L.table.copy()
    bad[1, 2] += 1  # pixel offset that is not the prefix sum of the sizes
    assert align(acfg, fake, bad.ctypes.data_as(ctypes.c_void_p)) == -1 and b"prefix" in lib.ddn_last_error_string()
    one_row = ViewLayout.from_shapes([(1, 60), (61, 33)])
    assert align(acfg, fake, one_row.host_ptr()) == -1  # the alignment needs H, W >= 2

    assert lib.ddn_build_pair_tables_ragged(2, 3, None, host, fake, fake, fake, fake, fake, None) == -1
    assert lib.ddn_build_pair_tables_ragged(3, 3, fake, host, fake, fake, fake, fake, fake, None) == -1  # V disagrees

    fcfg = _lib.FilterConfig()
    lib.ddn_filter_config_default(ctypes.byref(fcfg))

    def filt(cfg, layout, layout_host, k=3):
        return lib.ddn_backproject_filter_ragged(ctypes.byref(cfg), 2, k, layout, layout_host, fake, fake, fake, fake, 2, fake,
                                                 fake, None, None, None)

    assert filt(fcfg, None, host) == -1
    assert filt(fcfg, fake, host) == -1 and b"stride" in lib.ddn_last_error_string()  # layout built for stride 2
    fcfg.stride = 2
    assert filt(fcfg, fake, host, k=1025) == -1


def test_oracle_list_form_equals_array_form():
    """ragged_oracle.densify_views on per-view lists gives what restatement.densify gives on the [V,H,W] arrays of the same
    uniform scene."""
    sc = make_scene(SceneConfig(n_views=4, width=64, height=48, n_sparse=250, seed=5))
    poses, intr = sc.cam_from_world.numpy(), sc.intrinsics.numpy()
    nbr = nearest_views_table(poses, 2)
    arrays = (sc.mono_depth.numpy(), sc.normal.numpy(), sc.mask.numpy(), sc.rgb.numpy())
    kw = dict(align=R.AlignConfig(adaptive_correspondences=False), stride=2, voxel=0.05)
    a = R.densify(*arrays, sc.sparse_xyz.numpy(), sc.sparse_offsets.numpy(), poses, intr, nbr, 2, **kw)
    b = ragged_oracle.densify_views(*[list(x) for x in arrays], sc.sparse_xyz.numpy(), sc.sparse_offsets.numpy(), poses, intr, nbr, 2, **kw)
    assert isinstance(b["refined"], list) and np.array_equal(np.stack(b["refined"]), a["refined"])
    assert a["votes"].max() >= 1
    for k in ("points", "colors", "normals", "src_view", "pixel", "votes", "keep", "counts_per_view", "voxel_keys", "voxel_xyz",
              "voxel_rgb", "voxel_count", "active_views"):
        assert np.array_equal(a[k], b[k]), k
