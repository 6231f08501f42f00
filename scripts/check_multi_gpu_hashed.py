#!/usr/bin/env python
"""Multi-GPU equivalence check of the HASHED fusion path (run under torchrun on N GPUs of one node): scenes whose voxel
grid is too large for the sessions' dense occupancy bitmap - a dome background (SceneConfig.dome_radius) and a small
scene with a forced-small bitmap (max_grid_cells) - must come out of the N-rank sharded pipeline as out of the 1-rank
one, bit for bit (depthdensifier_b200/selfcheck.py), with and without N5 dedup, on even and uneven shards.  Rank 0
prints one JSON line.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
      scripts/check_multi_gpu_hashed.py
"""

import json
import os
import sys
from pathlib import Path

import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from depthdensifier_b200.selfcheck import multi_gpu_check  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    dist.init_process_group("nccl", device_id=dev)
    uneven = dict(n_views=29, width=203, height=131, k=3, voxel=0.03)  # 29 views: the last shards are short or empty
    reports = [multi_gpu_check(dev, rank, world, dome_radius=150.0),
               multi_gpu_check(dev, rank, world, dome_radius=150.0, dedup=True, **uneven),
               multi_gpu_check(dev, rank, world, max_grid_cells=1 << 16),
               multi_gpu_check(dev, rank, world, max_grid_cells=1 << 16, dedup=True, **uneven)]
    if rank == 0:
        print(json.dumps({"multi_gpu_check_hashed": reports}))
    dist.barrier()
    dist.destroy_process_group()
    ok = all(r["passed"] and r.get("grid") == "hashed" for r in reports)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
