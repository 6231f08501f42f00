"""The reprojection bound's argument checks, without a GPU: ops' support tuple, DensifyConfig, the CLI flag and the C
entry points."""

import ctypes as C
import math

import pytest

from depthdensifier_b200 import ops
from depthdensifier_b200.engine import DensifyConfig

BAD = [0.0, -1.0, math.inf, math.nan]


def test_support_tuple():
    assert ops._support_args((2, 0.01)) == (2, 0.01, None)
    assert ops._support_args((2, 0.01, 1)) == (2, 0.01, 1.0)
    for rho in BAD:
        with pytest.raises(ValueError):
            ops._support_args((2, 0.01, rho))
    with pytest.raises(ValueError):
        ops._support_args((2, 0.01, 1.0, 3))


def test_densify_config():
    assert DensifyConfig(min_support=2).support() == (2, 0.01)
    assert DensifyConfig(min_support=2, support_tau=0.02, support_reproj_px=1).support() == (2, 0.02, 1.0)
    assert DensifyConfig().support() is None
    with pytest.raises(ValueError):
        DensifyConfig(support_reproj_px=1.0)
    for rho in BAD:
        with pytest.raises(ValueError):
            DensifyConfig(min_support=1, support_reproj_px=rho)
    cfg = DensifyConfig(min_support=1)
    cfg.support_reproj_px = -2.0  # set after construction: support() still refuses it
    with pytest.raises(ValueError):
        cfg.support()


def test_cli_flag():
    tyro = pytest.importorskip("tyro")
    from depthdensifier_b200 import pipeline as P

    cfg = tyro.cli(P.ScriptConfig, args=["--filtering.min-support", "2", "--filtering.support-reproj-px", "0.5"])
    assert cfg.filtering.support_reproj_px == 0.5
    assert tyro.cli(P.ScriptConfig, args=[]).filtering.support_reproj_px is None


def test_entry_points_reject_bad_rho():
    from depthdensifier_b200 import _lib

    lib = _lib.load()
    cfg = ops.FilterOptions().to_c()
    for rho in BAD:
        rc = lib.ddn_backproject_filter_support_reproj(C.byref(cfg), 4, 0, 4, 8, 8, 2, None, None, None, None, None, 2, 1, 0.01,
                                                       rho, None, None, None, None, None, None)
        assert rc != 0 and b"reproj_px" in lib.ddn_last_error_string()
        rc = lib.ddn_backproject_filter_support_reproj_ragged(C.byref(cfg), 4, 2, None, None, None, None, None, None, 2, 1, 0.01,
                                                              rho, None, None, None, None, None, None)
        assert rc != 0 and b"reproj_px" in lib.ddn_last_error_string()
