"""The bucket plan of a one-GPU sort of 64-bit keys: k byte steps on the top bytes, then bucket_sort_kernel finishes
every run of equal top bytes on chip.  Every result is bit-exact against numpy's stable sort and identical to the byte
steps' (tune key bk_mode = 1); the stats match hostlogic's restatement of the plan -- needs a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
import key_orders as KO  # noqa: E402

TILE, C = 4096, 256  # BK_TILE, BK_C of csrc/lsb_bucket.cuh
NS = L.FLAG_NO_SKIP


@pytest.fixture
def bk():
    """lsb.tune of the bucket keys for one test, back at their defaults afterwards"""
    try:
        yield lsb.tune
    finally:
        lsb.tune("bk_mode", 0)
        lsb.tune("bk_bytes", 0)


def records(keys, vals=None):
    a = np.empty(len(keys), dtype=L.ELT)
    a["key"] = keys
    a["val"] = np.arange(len(keys), dtype=np.uint64) if vals is None else vals
    return a


def expected_stats(a, flags, mode=0, forced=0):
    """(subpasses, partition_launches, kernel_launches, skipped) the plan predicts for sorting `a`"""
    ok = KO.order_key(a["key"], flags)
    counts = H.byte_counts(ok)
    n = len(a)
    k = H.bucket_plan(counts, n, no_skip=bool(flags & NS), mode=mode, forced=forced)
    skipped = 0 if k or flags & NS else int((counts == n).any(axis=1).sum())
    return H.sort_stats(k, k and overflows(ok, k), skipped) + (skipped,)


def overflows(ok, k):
    """a bucket of the top 8k bits holds more than C records whose order keys are not already in order"""
    top = ok >> np.uint64(64 - 8 * k)
    order = np.argsort(top, kind="stable")
    t, o = top[order], ok[order]
    starts = np.flatnonzero(np.r_[True, t[1:] != t[:-1]])
    ends = np.r_[starts[1:], len(t)]
    return any(bool((o[s + 1:e] < o[s:e - 1]).any()) for s, e in zip(starts, ends) if e - s > C)


def sort_once(tune, a, flags=0, mode=0, forced=0, how="sort"):
    tune("bk_mode", mode)
    tune("bk_bytes", forced)
    n = len(a)
    with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
        if how == "sort":
            s.upload(a)
            st = s.my_sort()
            out = s.download()
        else:
            out = np.empty_like(a)
            st = s.sort_host(np.ascontiguousarray(a), out)
    return out, st


def check(tune, a, flags=0, mode=0, forced=0, how="sort"):
    want = KO.reference(a, flags)
    got, st = sort_once(tune, a, flags, mode, forced, how)
    assert (got == want).all()
    sub, launches, kernels, skipped = expected_stats(a, flags, mode, forced)
    assert (st.subpasses, st.partition_launches, st.kernel_launches, st.skipped) == (sub, launches, kernels, skipped)
    assert st.partition_elements == launches * len(a)
    ref, st1 = sort_once(tune, a, flags, 1, 0, how)
    assert ref.tobytes() == got.tobytes()
    return st


def uniform(n, seed):
    return np.random.default_rng(seed).integers(0, 1 << 64, size=n, dtype=np.uint64, endpoint=False)


@pytest.mark.parametrize("n", [1 << 20, (1 << 23) + 1])
@pytest.mark.parametrize("flags", [0, NS])
def test_uniform_keys_take_the_plan(bk, n, flags):
    a = records(uniform(n, n))
    st = check(bk, a, flags)
    k = H.bucket_bytes(n)
    assert (st.subpasses, st.partition_launches) == (8, k + 1)


@pytest.mark.parametrize("n", [1, 2, 31, 257, TILE - 1, TILE, TILE + 1, TILE + C - 1, TILE + C, TILE + C + 1,
                               TILE + C + 2, 3 * TILE + 100])
@pytest.mark.parametrize("k", [2, 3, 4])
def test_ragged_sizes(bk, n, k):
    a = records(uniform(n, 7 * n + k))
    a["key"][n // 3:n // 3 + n // 4] = a["key"][0]  # a run of equal keys: where they meet, stability decides
    check(bk, a, NS, mode=2, forced=k)


def f64_mix(n, seed):
    """uniform double bit patterns without NaNs (they would all share one bucket), plus 100 special values"""
    rng = np.random.default_rng(seed)
    k = uniform(n, seed)
    nan_or_inf = ((k >> np.uint64(52)) & np.uint64(0x7FF)) == np.uint64(0x7FF)
    k[nan_or_inf] ^= np.uint64(1 << 62)
    k[rng.integers(0, n, 100)] = KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), 100)]
    return k


@pytest.mark.parametrize("order", sorted(KO.ORDERS))
@pytest.mark.parametrize("how", ["sort", "host"])
def test_key_orders(bk, order, how):
    flags = KO.ORDERS[order]
    n = (1 << 20) + 77
    a = records(f64_mix(n, 11))
    st = check(bk, a, flags, how=how)
    assert st.subpasses == 8 and st.partition_launches == 3


@pytest.mark.parametrize("order", sorted(KO.ORDERS))
def test_key_orders_sort_device(order):
    torch = pytest.importorskip("torch")
    flags = KO.ORDERS[order]
    n = (1 << 20) + 77
    keys = f64_mix(n, 12)
    with lsb.DistributedSorter(n, ranks=1, flags=flags) as s:
        kt = torch.from_numpy(KO.typed(keys, flags).copy()).cuda()
        ko, vo, st = s.sort_device(kt)
        torch.cuda.synchronize()
    idx = KO.argsort(keys, flags)
    assert (vo.cpu().numpy() == idx).all()
    assert (ko.cpu().numpy().view(np.uint64) == keys[idx]).all()
    assert st.subpasses == 8 and st.partition_launches == 3


@pytest.mark.parametrize("order", ["f64", "f64_desc"])
def test_nan_bucket_longer_than_a_chunk(bk, order):
    # uniform bits read as doubles: ~n / 2048 NaNs share one order key, a bucket of ~512 records that is already in order
    n = (1 << 20) + 7
    a = records(uniform(n, 9))
    assert not overflows(KO.order_key(a["key"], KO.ORDERS[order]), 2)
    st = check(bk, a, KO.ORDERS[order] | NS)
    assert (st.subpasses, st.partition_launches, st.kernel_launches) == (8, 3, 5)


def test_long_runs_already_in_order_are_copied(bk):
    # two buckets longer than a chunk whose records are in order in the input: one repeated key over 900 records, and
    # ascending low bits over three tiles; both are copied through, no overflow
    rng = np.random.default_rng(13)
    n = 6 * TILE
    keys = uniform(n, 13)
    perm = rng.permutation(n)
    run1, run2 = np.sort(perm[:900]), np.sort(perm[900:900 + 3 * TILE])
    keys[run1] = np.uint64(0xAAAAAA << 40 | 5)
    keys[run2] = np.uint64(0x555555 << 40) | np.sort(rng.integers(0, 1 << 40, len(run2), dtype=np.uint64))
    a = records(keys)
    assert not overflows(a["key"], 3)
    st = check(bk, a, NS, mode=2, forced=3)
    assert (st.subpasses, st.partition_launches) == (8, 4)


def bucketed(sizes, k, seed, low_values=None):
    """records whose top 8k bits form buckets of the given sizes in order (distinct tops, increasing), shuffled"""
    rng = np.random.default_rng(seed)
    nb = len(sizes)
    pool = np.unique(rng.integers(0, 1 << (8 * k), size=2 * nb, dtype=np.uint64))
    tops = np.sort(pool[rng.choice(len(pool), nb, replace=False)])
    top = np.repeat(tops, sizes)
    n = len(top)
    low_bits = 64 - 8 * k
    if low_values is None:
        low = rng.integers(0, 1 << low_bits, size=n, dtype=np.uint64)
    else:
        low = rng.choice(np.asarray(low_values, dtype=np.uint64), n)
    keys = top << np.uint64(low_bits) | low
    return records(keys[rng.permutation(n)])


def test_buckets_at_the_chunk_capacity(bk):
    sizes = [C, 1, C, C - 1, 3] * 40
    st = check(bk, bucketed(sizes, 3, 1), NS, mode=2, forced=3)
    assert st.subpasses == 8


def test_a_bucket_over_the_capacity_falls_back(bk):
    sizes = [5] * 1000 + [C + 1] + [5] * 1000
    st = check(bk, bucketed(sizes, 3, 2), NS, mode=2, forced=3)
    assert (st.subpasses, st.partition_launches) == (3 + 8, 3 + 9)


def test_buckets_across_tile_and_halo_edges(bk):
    # buckets of 200: every tile boundary and every halo end cuts one, at a different offset per tile
    sizes = [200] * ((6 * TILE) // 200) + [1] * 57 + [200] * 60
    check(bk, bucketed(sizes, 3, 3), NS, mode=2, forced=3)
    # the last bucket of a tile as long as the halo allows
    sizes = [1] * (TILE - 1) + [C] + [1] * 300
    check(bk, bucketed(sizes, 3, 4), NS, mode=2, forced=3)


def test_chunks_of_256_one_record_buckets(bk):
    check(bk, bucketed([1] * (8 * TILE + 3), 2, 5), NS, mode=2, forced=2)


def test_duplicate_keys_in_one_bucket(bk):
    sizes = [C, 100, C, 17] * 30
    check(bk, bucketed(sizes, 4, 6, low_values=[0, 1, 0xFFFFFFFF]), NS, mode=2, forced=4)


@pytest.mark.parametrize("flags", [0, NS])
def test_correlated_top_bytes_fall_back(bk, flags):
    # top three bytes (b, b, b): every byte histogram is uniform, but each top-16-bit bucket holds n / 256 records
    n = 1 << 21
    keys = uniform(n, 9)
    b = keys >> np.uint64(56)
    keys = (b << np.uint64(56)) | (b << np.uint64(48)) | (b << np.uint64(40)) | (keys & np.uint64((1 << 40) - 1))
    a = records(keys)
    st = check(bk, a, flags)
    assert (st.subpasses, st.partition_launches) == (2 + 8, 2 + 9)


@pytest.mark.parametrize("mask,draws", [(0xFFFFFF, 1), (0xFFFFFFFFFFFFFFFF, 3)])
def test_skewed_keys_decline(bk, mask, draws):
    n = 1 << 21
    rng = np.random.default_rng(10)
    keys = uniform(n, 10) & np.uint64(mask)
    for _ in range(draws - 1):
        keys &= rng.integers(0, 1 << 64, size=n, dtype=np.uint64, endpoint=False)
    st = check(bk, records(keys), 0)
    assert st.partition_launches == st.subpasses  # the byte steps
