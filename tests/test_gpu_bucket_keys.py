"""The chunk keys of bucket_sort_kernel: a chunk is sorted by a 32-bit key (bucket ordinal, a prefix of the low bits,
position) and again by the 64-bit key when two of its records share ordinal and prefix but not their order keys.
Inputs where every chunk, some chunks or no chunk takes the 64-bit sort, the widest ordinal, k = 2 and 3, runs of ties
in buckets at and past the chunk capacity, all four 64-bit orders and radix 8 and 16.  Every result is bit-exact
against numpy's stable sort and identical to the byte steps' (tune key bk_mode = 1); the stats match hostlogic's
restatement of the plan -- needs a B200."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import distributed_lsb_b200 as lsb  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
import key_orders as KO  # noqa: E402

C = 256  # BK_C of csrc/lsb_bucket.cuh
NS = L.FLAG_NO_SKIP
U64 = np.uint64


@pytest.fixture
def tune_bk():
    """lsb.tune of the bucket keys for one test, back at their defaults afterwards"""
    try:
        yield lsb.tune
    finally:
        lsb.tune("bk_mode", 0)
        lsb.tune("bk_bytes", 0)


def raw_keys(ok, flags):
    """raw 64-bit patterns whose order key under `flags` is `ok` (up to NaN patterns, which all share one)"""
    k = np.asarray(ok, dtype=U64).copy()
    if flags & KO.DESC:
        k = ~k
    if flags & KO.F64:
        pos = (k & KO.TOP) != 0
        k = np.where(pos, k ^ KO.TOP, ~k)
    elif flags & KO.I64:
        k = k ^ KO.TOP
    return k


def records(keys):
    a = np.empty(len(keys), dtype=L.ELT)
    a["key"] = keys
    a["val"] = np.arange(len(keys), dtype=U64)
    return a


def overflows(ok, k):
    top = ok >> U64(64 - 8 * k)
    order = np.argsort(top, kind="stable")
    t, o = top[order], ok[order]
    starts = np.flatnonzero(np.r_[True, t[1:] != t[:-1]])
    ends = np.r_[starts[1:], len(t)]
    return any(bool((o[s + 1:e] < o[s:e - 1]).any()) for s, e in zip(starts, ends) if e - s > C)


def run(tune, a, flags, mode, forced, radix):
    tune("bk_mode", mode)
    tune("bk_bytes", forced)
    with lsb.DistributedSorter(len(a), ranks=1, flags=flags, radix_bits=radix) as s:
        s.upload(a)
        st = s.my_sort()
        return s.download(), st


def check(tune, a, flags=NS, mode=2, forced=0, radix=16, expect_k=None):
    """sorts `a` with the bucket plan and with the byte steps; both must equal numpy's stable sort"""
    got, st = run(tune, a, flags, mode, forced, radix)
    want = KO.reference(a, flags)
    assert got.tobytes() == want.tobytes()
    ok = KO.order_key(a["key"], flags)
    n = len(a)
    k = H.bucket_plan(H.byte_counts(ok), n, radix_bits=radix, no_skip=bool(flags & NS), mode=mode, forced=forced)
    if expect_k is not None:
        assert k == expect_k
    skipped = 0 if k or flags & NS else int((H.byte_counts(ok) == n).any(axis=1).sum())
    assert (st.subpasses, st.partition_launches, st.kernel_launches) == H.sort_stats(k, k and overflows(ok, k), skipped)
    ref, _ = run(tune, a, flags, 1, 0, radix)
    assert ref.tobytes() == got.tobytes()


def bucketed(sizes, k, rng, low):
    """order keys: buckets of the given sizes on distinct increasing tops of 8k bits, low parts low(rng, top, size)"""
    nb = len(sizes)
    pool = np.unique(rng.integers(0, 1 << (8 * k), size=2 * nb, dtype=U64))
    tops = np.sort(pool[rng.choice(len(pool), nb, replace=False)])
    lb = U64(64 - 8 * k)
    parts = [t << lb | low(rng, i, s) for i, (t, s) in enumerate(zip(tops, sizes))]
    ok = np.concatenate(parts)
    return ok[rng.permutation(len(ok))]


ORDER_IDS = ["u64", "i64", "f64", "u64_desc"]


@pytest.mark.parametrize("order", ORDER_IDS)
@pytest.mark.parametrize("radix", [8, 16])
def test_every_chunk_falls_back(tune_bk, order, radix):
    # top 3 bytes spread, next 3 constant, low 2 random: the prefix of every 32-bit key is the constant, so every chunk
    # has ties that the 64-bit key must order
    flags = KO.ORDERS[order] | NS
    rng = np.random.default_rng(1)
    n = (1 << 21) + 3
    top = rng.integers(0, 1 << 14, n, dtype=U64) << U64(10)  # 2^14 buckets spread over the top 3 bytes, ~128 records each
    ok = top << U64(40) | U64(0x3C3C3C << 16) | rng.integers(0, 1 << 16, n, dtype=U64)
    check(tune_bk, records(raw_keys(ok, flags)), flags, forced=3, radix=radix, expect_k=3)


@pytest.mark.parametrize("order", ORDER_IDS)
def test_some_chunks_fall_back(tune_bk, order):
    # k = 3 (40 low bits): half the buckets draw their low parts from three values that differ only in the last bits
    # (ties of the prefix with different order keys), the other half from three values far apart (equal keys only)
    flags = KO.ORDERS[order] | NS
    rng = np.random.default_rng(2)
    sizes = rng.integers(1, 120, 20000)

    def low(rng, i, s):
        base = rng.integers(0, 1 << 39, dtype=U64)
        vals = base + np.array([0, 1, 5], dtype=U64) if i % 2 else np.array([0, 1 << 30, 1 << 38], dtype=U64) + base
        return rng.choice(vals, s)

    check(tune_bk, records(raw_keys(bucketed(sizes, 3, rng, low), flags)), flags, forced=3)


@pytest.mark.parametrize("order", ORDER_IDS)
def test_no_chunk_falls_back_exact_prefix(tune_bk, order):
    # k = 7: the low part is one byte and always fits the prefix; buckets of several records with repeated low bytes
    flags = KO.ORDERS[order] | NS
    rng = np.random.default_rng(3)
    sizes = rng.integers(2, 40, 60000)
    check(tune_bk, records(raw_keys(bucketed(sizes, 7, rng, lambda r, i, s: r.integers(0, 256, s, dtype=U64)), flags)),
          flags, forced=7)


@pytest.mark.parametrize("radix", [8, 16])
def test_widest_ordinal(tune_bk, radix):
    # k = 7 at 2^20 records, nearly all buckets singletons: chunks of 256 one-record buckets (ordinal 0..255, 8 bits)
    rng = np.random.default_rng(4)
    n = 1 << 20
    ok = np.unique(rng.integers(0, 1 << 64, n + 4096, dtype=U64, endpoint=False))[:n]
    ok = ok[rng.permutation(n)]
    ok[rng.integers(0, n, 64)] = ok[0]  # a few repeats
    check(tune_bk, records(ok), NS, forced=7, radix=radix)


@pytest.mark.parametrize("order", ORDER_IDS)
def test_k2_at_2_21(tune_bk, order):
    # the plan's own k: 2 at 2^21 records (48 low bits, prefix of 22 or fewer), byte counts uniform
    flags = KO.ORDERS[order]
    rng = np.random.default_rng(5)
    n = 1 << 21
    ok = rng.integers(0, 1 << 64, n, dtype=U64, endpoint=False)
    m = n // 8  # prefix ties with equal and with different keys
    ok[:m] = (ok[:m] & ~U64((1 << 46) - 1)) | rng.choice(np.array([77, 78, 1 << 30], dtype=U64), m)
    keys = raw_keys(ok, flags)
    if flags & KO.F64:
        keys[rng.integers(0, n, 200)] = KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), 200)]
    check(tune_bk, records(keys), flags, mode=0, expect_k=2)


@pytest.mark.parametrize("order", ["u64", "f64_desc"])
def test_k3_above_2_23(tune_bk, order):
    flags = KO.ORDERS[order]
    rng = np.random.default_rng(6)
    n = (1 << 23) + 1000
    keys = raw_keys(rng.integers(0, 1 << 64, n, dtype=U64, endpoint=False), flags)
    if flags & KO.F64:
        keys[rng.integers(0, n, 500)] = KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), 500)]
    check(tune_bk, records(keys), flags, mode=0, expect_k=3)


@pytest.mark.parametrize("size", [C, C + 1])
@pytest.mark.parametrize("order", ORDER_IDS)
def test_tie_runs_in_full_and_overfull_buckets(tune_bk, size, order):
    # buckets of exactly 256 and 257 records made of runs of equal keys and of keys equal in the prefix only;
    # a 257-record bucket out of order overflows into the byte steps
    flags = KO.ORDERS[order] | NS
    rng = np.random.default_rng(7)
    sizes = [size, 3, size, 40, 1] * 30

    def low(rng, i, s):
        base = rng.integers(0, 1 << 38, dtype=U64)
        return base + rng.choice(np.array([0, 0, 0, 2, 2, 1 << 20, 9], dtype=U64), s)

    check(tune_bk, records(raw_keys(bucketed(sizes, 3, rng, low), flags)), flags, forced=3)


def test_f64_nans_and_signed_zeros(tune_bk):
    # uniform doubles with NaNs of both signs, ±inf and ±0 among them: NaNs share one order key (one bucket already in
    # order), -0.0 and +0.0 share one and meet the smallest positive doubles
    flags = KO.F64 | NS
    rng = np.random.default_rng(8)
    n = (1 << 21) + 11
    keys = raw_keys(rng.integers(0, 1 << 64, n, dtype=U64, endpoint=False), flags)
    keys[rng.integers(0, n, 2000)] = KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), 2000)]
    zero = rng.integers(0, n, 2000)
    keys[zero] = rng.integers(0, 2, 2000, dtype=U64) << U64(63)
    keys[rng.integers(0, n, 2000)] = rng.integers(1, 1 << 12, 2000, dtype=U64)  # denormals next to +0
    check(tune_bk, records(keys), flags, forced=3)
