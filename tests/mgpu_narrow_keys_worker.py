"""Worker for tests/test_multigpu_narrow_keys.py: one process per GPU (torchrun).  Each rank passes CUDA tensors of its
`here` narrow keys to a sorter made with key_dtype (lsb_sort_device_typed) and checks its slice [first_global,
first_global + here) of numpy's stable argsort of the typed values, the values being global input indices.  Exit code
0 == all passed."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import distributed_lsb_b200 as lsb  # noqa: E402
import narrow_keys as NK  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402


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
        for name in ("float32", "bfloat16", "int16", "uint32"):
            bits = NK.special_mix(n, name, seed=seed)
            for descending in (False, True):
                for shape in (0, L.FLAG_ONE_PASS):
                    flags = shape | (L.FLAG_DESCENDING if descending else 0)
                    s = make(n, rank, world, device, flags=flags, key_dtype=NK.torch_dtype(torch, name))
                    lo, hi = s.first_global, s.first_global + s.here
                    k, v, st = s.sort_device(NK.to_device(torch, bits[lo:hi], name))
                    perm = NK.argsort(bits, name, descending)
                    what = (name, descending, shape, n)
                    assert np.array_equal(NK.bits_of(torch, k), bits[perm][lo:hi]), what
                    assert np.array_equal(v.cpu().numpy(), perm[lo:hi]), what
                    assert st.passes == NK.BITS[name] // 16, what
                    s.close()
    dist.barrier()
    dist.destroy_process_group()
    print(f"rank {rank}/{world}: multi-GPU narrow-key sort ok")


if __name__ == "__main__":
    main()
