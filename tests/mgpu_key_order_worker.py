"""Worker for tests/test_multigpu_key_order.py: one process per GPU (torchrun).  Each rank sorts its shard of keys
read as float64 and as int64, ascending and descending, and checks its slice against numpy's stable argsort of the
typed view; verify() must pass globally (the cross-shard comparison uses the order).  Exit code 0 == all passed."""
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
from oracle import oracle as O  # noqa: E402


def make(n, rank, world, **kw):
    s = lsb.DistributedSorter(n, ranks=world, world_size=world, world_rank=rank,
                              device=int(os.environ.get("LOCAL_RANK", "0")), **kw)
    ids = [lsb.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    s.comm_init(ids[0])
    return s


def check(s, a, korder, what):
    lo, hi = s.first_global, s.first_global + s.here
    want = KO.reference(a, korder)
    got = s.download()
    assert np.array_equal(got.view(np.uint64), want[lo:hi].view(np.uint64)), what
    v = s.verify()
    assert v.order_violations == 0 and v.elements == len(a) and list(v.checksum) == O.checksum(a), what


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0"))))
    n = (1 << 21) + 12345
    g = O.generate(n, world)[:n]  # pcg64 keys, read as doubles (NaNs included) and as int64
    for order in ("f64", "f64_desc", "i64", "i64_desc"):
        for shape in (0, L.FLAG_ONE_PASS):
            korder = KO.ORDERS[order]
            s = make(n, rank, world, flags=korder | shape)
            s.generate()
            s.my_sort()
            check(s, g, korder, (order, shape))
            s.close()
    # an uploaded special-value mix: ties between -0.0 / +0.0 and between NaNs run across shard boundaries
    m = (1 << 20) + 77
    a = np.zeros(m, dtype=L.ELT)
    a["key"] = KO.special_mix(m, seed=1)
    a["val"] = np.arange(m, dtype=np.uint64)
    for order in ("f64", "f64_desc"):
        s = make(m, rank, world, flags=KO.ORDERS[order])
        s.upload(a[s.first_global:s.first_global + s.here])
        s.my_sort()
        check(s, a, KO.ORDERS[order], ("special", order))
        s.close()
    dist.barrier()
    dist.destroy_process_group()
    print(f"rank {rank}/{world}: multi-GPU key order ok")


if __name__ == "__main__":
    main()
