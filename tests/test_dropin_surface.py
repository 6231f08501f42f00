"""The drop-in surface: names, parameter lists and defaults of the reference's entry points are kept (compared
against the reference's surface, recorded in tests/golden/ref_surface.json by oracle/make_golden.py), and the tyro
CLI renders the same flags."""

import json
import subprocess
import sys

import pytest

from oracle.make_golden import _defaults, _params, batch_output_dir


@pytest.fixture(scope="module")
def ref(golden_dir):
    return json.loads((golden_dir / "ref_surface.json").read_text())


def test_depth_refiner_surface_matches_reference(ref):
    from depthdensifier_b200 import DepthRefiner, RefinerConfig

    assert _defaults(RefinerConfig) == ref["RefinerConfig"]
    mine, theirs = _params(DepthRefiner.__init__), ref["DepthRefiner.__init__"]
    assert mine[: len(theirs)] == theirs  # extras (align_mode, subsample_seed, device) are keyword-only additions
    assert _params(DepthRefiner.refine_depth)[:6] == ref["DepthRefiner.refine_depth"]


def test_script_config_tree_matches_reference(ref):
    from depthdensifier_b200 import pipeline as P

    for name in ("PathsConfig", "MoGeConfig", "ProcessingConfig", "FilteringConfig"):
        mine, theirs = _defaults(getattr(P, name)), ref[name]
        assert {k: mine[k] for k in theirs} == theirs, name  # every reference field, same default
    assert set(ref["ScriptConfig"]) <= set(_defaults(P.ScriptConfig))
    assert _params(P.project_points) == ref["project_points"]
    assert _params(P.unproject_points) == ref["unproject_points"]
    assert _params(P.main)[:1] == ref["main"] == ["config"]


def test_fast_pchip_surface_matches_reference(ref):
    from depthdensifier_b200 import fast_pchip_refiner as mine

    assert _defaults(mine.FastPCHIPRefinerConfig) == ref["FastPCHIPRefinerConfig"]
    theirs = ref["FastPCHIPRefiner.__init__"]
    assert _params(mine.FastPCHIPRefiner.__init__)[: len(theirs)] == theirs
    assert _params(mine.FastPCHIPRefiner.refine_depth) == ref["FastPCHIPRefiner.refine_depth"]
    assert _params(mine.refine_depth_from_colmap) == ref["refine_depth_from_colmap"]


def test_gradient_mask_signature_matches_reference(ref):
    import inspect

    from depthdensifier_b200.edge_masks import compute_depth_normal_gradient_mask

    a = inspect.signature(compute_depth_normal_gradient_mask)
    assert [[p.name, repr(p.default)] for p in a.parameters.values()] == ref["compute_depth_normal_gradient_mask"]


def test_batch_config_matches_reference(ref, tmp_path):
    """scripts/run_batch.py: same BatchConfig fields (root_dir and output_dir required, the ScriptConfig embedded as
    `config`), and each scan's model goes to <output_dir>/<scan>/sparse/0 (scripts/run_batch.py:63-65)."""
    import dataclasses

    from depthdensifier_b200 import run_batch as mine

    theirs = [tuple(f) for f in ref["BatchConfig"]]
    ours = [(f.name, f.default is dataclasses.MISSING and f.default_factory is dataclasses.MISSING) for f in dataclasses.fields(mine.BatchConfig)]
    assert ours[: len(theirs)] == theirs  # root_dir (required), output_dir (required), config; additions follow
    # output layout: main over a root with one complete scan, densification itself stubbed out
    assert batch_output_dir(mine, tmp_path) == ref["batch_output_model_dir"] == "scan_a/sparse/0"


def test_package_exports():
    import depthdensifier_b200 as pkg

    assert pkg.__all__ == ["DepthRefiner", "RefinerConfig"] and pkg.__version__ == "0.1.0"  # src/depthdensifier/__init__.py:3-6


def test_cli_flags():
    """tyro renders the reference's flags (scripts/run_batch.py:36-37 names --filtering.vote-threshold)."""
    out = subprocess.run([sys.executable, "-m", "depthdensifier_b200.pipeline", "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-500:]
    for flag in ("--paths.recon-path", "--paths.image-dir", "--paths.output-model-dir", "--moge.checkpoint",
                 "--processing.pipeline-downsample-factor", "--processing.downsample-density", "--refiner.min-correspondences",
                 "--filtering.vote-threshold", "--filtering.depth-threshold", "--fusion.voxel-size", "--filtering.num-neighbours"):
        assert flag in out.stdout, flag
    out = subprocess.run([sys.executable, "-m", "depthdensifier_b200.run_batch", "--help"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "--root-dir" in out.stdout and "--output-dir" in out.stdout
    assert "--config.filtering.vote-threshold" in out.stdout  # the flag scripts/run_batch.py:36-37 documents
