#!/usr/bin/env python
"""The split large scenes of bench.py (C4 / C5 over the GPUs of a box through the library-owned NCCL communicator) on their own:

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P scripts/bench_large_only.py"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist
    import bench
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    out = bench.measure_large_scenes(local_rank, rank, world)
    if rank == 0:
        print(json.dumps({"n_gpus": world, "ms_per_eval": {k: v.get("ms_per_eval", v.get("error")) for k, v in out.items()}}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
