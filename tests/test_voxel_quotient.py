"""The voxel coordinate's division-free quotient (csrc/voxel_quotient.cuh) floors exactly as floorf(a / v) in IEEE
float32.  The header is compiled into a host program (tests/voxel_quotient_check.cpp) with g++, so this runs without a
GPU; the kernels include the same header."""

from __future__ import annotations

import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

HERE = Path(__file__).resolve().parent


@pytest.fixture(scope="module")
def checker(tmp_path_factory):
    cxx = shutil.which("g++")
    if cxx is None:
        pytest.skip("g++ not found")
    exe = tmp_path_factory.mktemp("vq") / "voxel_quotient_check"
    flags = ["-std=c++17", "-O2", "-ffp-contract=off", "-fopenmp"]
    # fmaf is exact with or without the FMA instruction; the instruction only makes the sweep faster
    cpuinfo = Path("/proc/cpuinfo")
    if cpuinfo.exists() and " fma " in cpuinfo.read_text():
        flags.append("-mfma")
    subprocess.run([cxx, *flags, "-o", str(exe), str(HERE / "voxel_quotient_check.cpp")], check=True)
    return exe


def _run(exe, *args):
    r = subprocess.run([str(exe), *map(str, args)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0 and " mismatches 0" in r.stdout, r.stdout
    return r.stdout


# the benchmark's voxel (0.01), the self-check's (0.03), a finer one and a coarse one with a periodic reciprocal
@pytest.mark.parametrize("voxel", [0.01, 0.03, 0.005, 1.0 / 3.0])
def test_every_float32(checker, voxel):
    bits = int(np.float32(voxel).view(np.uint32))
    out = _run(checker, "exhaustive", f"{bits:08x}")
    assert "checked 4294967296 " in out


def test_integer_boundaries(checker):
    # 200 voxel sizes in [1e-4, 10], plus 50 at significands just above 1 and just below 2; 129 floats around
    # each of the 2^22 boundaries k * v, 1 <= |k| <= 2^21
    out = _run(checker, "boundaries", 200, 20261020)
    assert f"checked {250 * 2 * (1 << 21) * 129} " in out
