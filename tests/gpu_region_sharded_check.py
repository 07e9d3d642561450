"""Run under torchrun (one rank per GPU): getTotalForDimensionItems, getDistribution and copyMeasureData of a
sharded cube on real devices over NCCL must match the unsharded cube (device stores) built on rank 0.
python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513
tests/gpu_region_sharded_check.py"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_region_queries import _sharded_collect, _sharded_dims, _sharded_fill, assert_same_outcome  # noqa: E402


def _same(key, g, w):
    if key[0] == "data":
        return np.allclose(g, w, rtol=0, atol=0, equal_nan=True)
    if key[0] == "copy":
        return g == w
    try:
        assert_same_outcome(g, w)
        return True
    except AssertionError:
        return False


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from olap_in_memory_b200 import Cube, _native
    from olap_in_memory_b200.sharded import ShardedCube

    _native.init(local)
    failures = 0
    for prefix in (1, 2):
        for diced in (False, True):
            cube = ShardedCube(_sharded_dims(), prefix=prefix)
            _sharded_fill(cube, 5)
            got = _sharded_collect(cube, diced)
            if rank == 0:
                one = Cube(_sharded_dims())
                _sharded_fill(one, 5)
                want = _sharded_collect(one, diced)
                for key in want:
                    if not _same(key, got[key], want[key]):
                        failures += 1
                        print("MISMATCH", prefix, diced, key, str(got[key])[:200], str(want[key])[:200])
    ShardedCube.release_peer_buffers()
    t = torch.tensor([failures], device="cuda")
    dist.all_reduce(t)
    if rank == 0:
        print(f"gpu_region_sharded_check: world={world} failures={int(t.item())} launches={_native.lib().olap_kernel_launches()}")
    dist.destroy_process_group()
    sys.exit(1 if int(t.item()) else 0)


if __name__ == "__main__":
    main()
