#!/usr/bin/env python
"""Multi-GPU equivalence check (run under torchrun on N GPUs of one node): the N-rank sharded pipeline must
reproduce the 1-rank pipeline bit for bit (depthdensifier_b200/selfcheck.py).  Rank 0 prints one JSON line.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 \
      scripts/check_multi_gpu.py [--min-support M [--support-reproj-px R]] [--fuse-normals]

--min-support M: run both checks with the multi-view support filter (DensifyConfig.min_support = M) as well.
--support-reproj-px R: those support checks also with the forward-backward reprojection test
(DensifyConfig.support_reproj_px = R).
--fuse-normals: also run the dense and the dedup check, and a check whose grid is too large for the sessions' bitmap (the
hashed merge), with fused normals (DensifyConfig.fuse_normals); the per-point and voxel normals must match too.
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
    ms = [None]
    if "--min-support" in sys.argv:
        ms.append(int(sys.argv[sys.argv.index("--min-support") + 1]))
    rho = float(sys.argv[sys.argv.index("--support-reproj-px") + 1]) if "--support-reproj-px" in sys.argv else None
    reports = []
    for m in ms:
        r = None if m is None else rho
        reports += [multi_gpu_check(dev, rank, world, min_support=m, support_reproj_px=r),
                    multi_gpu_check(dev, rank, world, n_views=29, width=203, height=131, k=3, voxel=0.03, dedup=True, min_support=m,
                                    support_reproj_px=r)]
    if "--fuse-normals" in sys.argv:
        reports += [multi_gpu_check(dev, rank, world, fuse_normals=True),
                    multi_gpu_check(dev, rank, world, n_views=29, width=203, height=131, k=3, voxel=0.03, dedup=True, fuse_normals=True),
                    multi_gpu_check(dev, rank, world, dome_radius=150.0, fuse_normals=True)]
    if rank == 0:
        print(json.dumps({"multi_gpu_check": reports}))
    dist.barrier()
    dist.destroy_process_group()
    sys.exit(0 if all(r["passed"] for r in reports) else 1)


if __name__ == "__main__":
    main()
