"""Multi-rank hardware test of the hashed fusion path (skipped below two GPUs): N-rank == 1-rank bit for bit over the
NVLink peer-memory path for grids too large for the dense bitmap, run as a real torchrun job
(scripts/check_multi_gpu_hashed.py)."""

import json
import socket
import subprocess
import sys
from pathlib import Path

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_hashed_ranks_equal_one_rank(lib_built):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    n = min(torch.cuda.device_count(), 4)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(ROOT / "scripts" / "check_multi_gpu_hashed.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=str(ROOT))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
    rep = json.loads(line)["multi_gpu_check_hashed"]
    assert all(r["passed"] for r in rep) and all(r["path"] == "peer" for r in rep) and all(r["grid"] == "hashed" for r in rep), rep
