"""A sort by two key columns past 2^31 elements through lsb.lexsort -- needs a B200 with the memory named in the skip.

int64 secondary and float32 primary at 2^31 + 2^20 + 7 elements: two rounds, so the second round's pack gathers the
primary at input indices past 2^31 that the records carry.  Checked with plain torch on the GPU, in chunks: the result
is a permutation, and (primary, secondary, index) strictly rises between neighbours.
"""
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import sort_check as C  # noqa: E402
from test_gpu_large import _room  # noqa: E402

BIG = (1 << 31) + (1 << 20) + 7


def test_two_rounds_past_2p31():
    n = BIG
    # columns 12 n, indices 8 n, the sorter's two shards 32 n, the permutation check n, chunk temporaries
    _room("lexsort of 2^31 + 2^20 + 7", 12 * n + 8 * n + 32 * n + n + 16 * 8 * C.CHUNK)
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    # few distinct values in both columns: the secondary decides most primary ties and the index decides the rest;
    # -0.0 beside +0.0 in the primary
    primary = torch.randint(-500, 500, (n,), device="cuda", generator=g, dtype=torch.int32).to(torch.float32)
    primary[torch.arange(0, n, 3, device="cuda")] = -0.0
    secondary = torch.randint(-(1 << 40), 1 << 40, (1 << 12,), device="cuda", generator=g)[
        torch.randint(0, 1 << 12, (n,), device="cuda", generator=g)]
    torch.cuda.empty_cache()  # the sorter's shards come from cudaMalloc, not from torch's cache
    idx = lsb.lexsort([secondary, primary])
    torch.cuda.empty_cache()
    assert idx.dtype == torch.int64 and idx.numel() == n
    seen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for lo in range(0, n, C.CHUNK):
        seen[idx[lo:lo + C.CHUNK]] = True
    assert bool(seen.all()) and int(idx.min()) == 0 and int(idx.max()) == n - 1
    del seen
    for lo in range(0, n - 1, C.CHUNK):
        hi = min(n, lo + C.CHUNK + 1)
        j = idx[lo:hi]
        p, s = primary[j], secondary[j]
        a, b = slice(0, -1), slice(1, None)
        rising = (p[a] < p[b]) | ((p[a] == p[b]) & ((s[a] < s[b]) | ((s[a] == s[b]) & (j[a] < j[b]))))
        assert bool(rising.all()), f"order violated in the chunk from {lo}"
        assert lo or bool((p[:1] == -500).all())
