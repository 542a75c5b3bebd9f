"""unique past 2^31 elements, sorted and consecutive -- needs a B200 with the memory named in the skip.

Checked on the device without a host sort, in chunks, by four properties that together define the answer: the values
strictly increase (sorted mode) or differ from their neighbour (consecutive mode); values[inverse] is order-equal to the
input; counts == bincount(inverse); index == the smallest position of every group (scatter_reduce amin).
"""
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import sort_check as C  # noqa: E402
from test_gpu_large import _room  # noqa: E402

BIG = (1 << 31) + (1 << 20) + 7


def _check(x, values, index, inverse, counts, consecutive):
    n, u = x.numel(), values.numel()
    assert index.numel() == u and counts.numel() == u and inverse.numel() == n
    a, b = values[:-1], values[1:]
    assert bool((a < b).all()) if not consecutive else bool((a != b).all())
    assert torch.equal(x[index], values)
    first = torch.full((u,), n, dtype=torch.int64, device="cuda")
    hist = torch.zeros(u, dtype=torch.int64, device="cuda")
    for lo in range(0, n, C.CHUNK):
        inv = inverse[lo:lo + C.CHUNK]
        assert torch.equal(values[inv], x[lo:lo + C.CHUNK]), f"values[inverse] differs in the chunk from {lo}"
        first.scatter_reduce_(0, inv, torch.arange(lo, lo + inv.numel(), device="cuda"), "amin")
        hist += torch.bincount(inv, minlength=u)
    assert torch.equal(hist, counts) and torch.equal(first, index)
    if consecutive:  # groups in input order: inverse rises by 0 or 1 between neighbours
        for lo in range(0, n - 1, C.CHUNK):
            hi = min(n - 1, lo + C.CHUNK)
            d = inverse[lo + 1:hi + 1] - inverse[lo:hi]
            assert bool(((d == 0) | (d == 1)).all())


@pytest.mark.parametrize("consecutive", [False, True])
def test_past_2p31(consecutive):
    n = BIG
    # the keys 8 n, index / inverse / counts 24 n, the sorter's two shards 32 n, the check's temporaries
    _room("unique of 2^31 + 2^20 + 7", 8 * n + 24 * n + 32 * n + 24 * C.CHUNK * 8)
    g = torch.Generator(device="cuda")
    g.manual_seed(11)
    # 2^24 distinct values: groups whose members lie on both sides of 2^31; runs of 64 equal keys in consecutive mode
    x = torch.randint(-(1 << 23), 1 << 23, (n,), device="cuda", generator=g)
    if consecutive:
        x = x[torch.arange(n, device="cuda") // 64]
    x[-1] = 1 << 40  # a group whose first occurrence is the last element
    torch.cuda.empty_cache()  # the sorter's shards come from cudaMalloc, not from torch's cache
    fn = lsb.unique_consecutive if consecutive else lsb.unique
    if consecutive:
        values, inverse, counts = fn(x, return_inverse=True, return_counts=True)
        index = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), counts.cumsum(0)[:-1]])
        assert index[-1] == n - 1
    else:
        values, index, inverse, counts = fn(x, return_index=True, return_inverse=True, return_counts=True)
        assert int(index[-1]) == n - 1
    torch.cuda.empty_cache()
    _check(x, values, index, inverse, counts, consecutive)
