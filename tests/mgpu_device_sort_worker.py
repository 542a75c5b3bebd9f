"""Worker for tests/test_multigpu_device_sort.py: one process per GPU (torchrun).  Each rank passes CUDA tensors of its
`here` keys to sort_device and checks its slice [first_global, first_global + here) of numpy's stable argsort of the
typed keys, the values being global input indices; verify() must pass globally.  Exit code 0 == all passed."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402

TORCH_DTYPE = {0: torch.uint64, KO.I64: torch.int64, KO.F64: torch.float64}


def make(n, rank, world, device, **kw):
    s = lsb.DistributedSorter(n, ranks=world, world_size=world, world_rank=rank, device=device, **kw)
    ids = [lsb.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    s.comm_init(ids[0])
    return s


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    device = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(device)
    dist.init_process_group("nccl", device_id=torch.device("cuda", device))
    for n, seed in (((1 << 21) + 12345, 1), (world * 3 + 1, 2)):  # the second: tiny shards, the last one shorter
        bits = KO.special_mix(n, seed=seed)
        for order in ("f64", "f64_desc", "i64", "i64_desc"):
            for shape in (0, L.FLAG_ONE_PASS):
                korder = KO.ORDERS[order]
                s = make(n, rank, world, device, flags=korder | shape)
                lo, hi = s.first_global, s.first_global + s.here
                keys = torch.from_numpy(bits[lo:hi].view(np.int64)).cuda().view(TORCH_DTYPE[korder & (KO.I64 | KO.F64)])
                k, v, _ = s.sort_device(keys)
                perm = KO.argsort(bits, korder)
                what = (order, shape, n)
                assert np.array_equal(k.view(torch.int64).cpu().numpy().view(np.uint64), bits[perm][lo:hi]), what
                assert np.array_equal(v.cpu().numpy(), perm[lo:hi]), what
                vf = s.verify()
                assert vf.order_violations == 0 and vf.elements == n, what
                s.close()
    dist.barrier()
    dist.destroy_process_group()
    print(f"rank {rank}/{world}: multi-GPU device sort ok")


if __name__ == "__main__":
    main()
