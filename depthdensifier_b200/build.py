"""In-tree build of libddn_b200.so (sm_100a only) with nvcc.  No JIT cache: the .so sits next to
the sources so it travels with the repo snapshot to the GPU box."""

from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libddn_b200.so"
SOURCES = ["api.cu", "align.cu", "filter.cu", "fuse.cu", "fuse_hash.cu", "fuse_hash_peers.cu", "geometry.cu", "pchip.cu", "masks.cu"]
NVCC_FLAGS = [
    "-std=c++17",
    "-O3",
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "--fmad=true",
    "-Xcompiler",
    "-fPIC,-O3,-fvisibility=hidden",
    "-Xptxas",
    "-v",
]


def nvcc_path() -> str:
    cand = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(cand):
        raise RuntimeError("nvcc not found; libddn_b200.so cannot be built (there is no CPU fallback)")
    return cand


def needs_build() -> bool:
    if not LIB_PATH.exists():
        return True
    t = LIB_PATH.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "ddn_b200.h"]
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False, suffix: str = "") -> Path:
    """``suffix``: build a variant next to the product library (libddn_b200<suffix>.so, own object directory) with
    the flags in $DDN_NVCC_EXTRA, e.g. -DDDN_K4_MINBLOCKS=4; load it with DDN_LIB_PATH.  Tuning experiments only."""
    lib_path = LIB_PATH if not suffix else PKG_DIR / f"libddn_b200{suffix}.so"
    if not suffix and not force and not needs_build():
        return LIB_PATH
    nvcc = nvcc_path()
    extra = os.environ.get("DDN_NVCC_EXTRA", "").split()
    objs = []
    build_dir = PKG_DIR / ("build" + suffix)
    build_dir.mkdir(exist_ok=True)
    log = []
    procs = []
    for src in SOURCES:
        obj = build_dir / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", str(CSRC / src), "-o", str(obj)]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, obj, pr in procs:
        out, _ = pr.communicate()
        log.append(f"== {src}\n{out}")
        if pr.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(str(obj))
    (build_dir / "ptxas.log").write_text("\n".join(log))
    cmd = [nvcc, "-shared", "-o", str(lib_path), *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    if verbose:
        print("\n".join(log))
    return lib_path


if __name__ == "__main__":
    sfx = next((a.split("=", 1)[1] for a in sys.argv if a.startswith("--suffix=")), "")
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv, suffix=sfx)
    print(p)
