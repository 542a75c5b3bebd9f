"""int64, float64 and descending key orders (include/lsbsort.h) through every pass shape -- needs a B200.

Whole sorts are compared record for record, bit for bit, with numpy's stable argsort of the typed view of the keys
(tests/key_orders.py), which shares no code with order_key.  Digit-level expectations (counts, starts, skips, the array
after one pass) come from the C oracle and the numpy restatement of order_key applied to the keys.
"""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import patterns as P  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from oracle import oracle as O  # noqa: E402
from test_gpu_patterns import _assert_same, _expected_skips  # noqa: E402

TL, OP, NS = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP
SHAPES = [0, NS, TL, OP, OP | NS, TL | OP]
SIZES = [P.PART_TILE + 1, P.SUPERTILE - 1, P.SUPERTILE + 1, (1 << 20) + 7]
ORDERS = ["u64_desc", "i64", "i64_desc", "f64", "f64_desc"]
F64_ORDERS = ["f64", "f64_desc"]
I64_ORDERS = ["i64", "i64_desc"]


def _records(keys):
    a = np.zeros(len(keys), dtype=P.ELT)
    a["key"] = keys
    a["val"] = np.arange(len(keys), dtype=np.uint64)
    return a


def _mixed(n, seed):
    """random bits, special values (both as doubles and as int64 extremes) and a few repeated keys: ties everywhere"""
    rng = np.random.default_rng([seed, n])
    k = rng.integers(0, 1 << 64, n, dtype=np.uint64)
    r = rng.random(n)
    sel = r < 0.3
    k[sel] = KO.SPECIAL_BITS[rng.integers(0, len(KO.SPECIAL_BITS), int(sel.sum()))]
    sel = (r >= 0.3) & (r < 0.5)
    k[sel] = rng.standard_normal(int(sel.sum())).view(np.uint64)
    sel = r >= 0.9
    k[sel] = rng.integers(0, 1 << 64, 7, dtype=np.uint64)[rng.integers(0, 7, int(sel.sum()))]
    return k


# f64 special-value mixes and int64 heavy hitters
def _zeros(rng, n):  # 90 % zeros, -0.0 and +0.0 interleaved: equal under the order, different bits
    k = rng.standard_normal(n).view(np.uint64)
    z = rng.random(n) < 0.9
    k[z] = np.where(rng.random(int(z.sum())) < 0.5, np.uint64(0), np.uint64(1 << 63))
    return k


def _nans(rng, n):  # NaNs with distinct payloads and both signs among normals
    k = rng.standard_normal(n).view(np.uint64)
    m = rng.random(n) < 0.3
    pay = rng.integers(1, 1 << 52, int(m.sum()), dtype=np.uint64)
    k[m] = np.uint64(0x7FF0000000000000) | pay | (rng.integers(0, 2, int(m.sum()), dtype=np.uint64) << np.uint64(63))
    return k


def _infs(rng, n):  # runs of +inf and -inf between normals
    k = rng.standard_normal(n).view(np.uint64)
    for start in range(0, n, 4096):
        if (start // 4096) % 3 == 0:
            k[start:start + 1000] = 0x7FF0000000000000 if (start // 4096) % 2 else 0xFFF0000000000000
    return k


def _normal(rng, n):  # a narrow exponent range: the high digits are nearly constant
    return rng.standard_normal(n).view(np.uint64)


def _i64_heavy(rng, n):  # INT64_MIN / INT64_MAX heavy hitters and values around 0
    k = rng.integers(-1000, 1000, n, dtype=np.int64).view(np.uint64)
    r = rng.random(n)
    k[r < 0.3] = 1 << 63
    k[(r >= 0.3) & (r < 0.6)] = (1 << 63) - 1
    return k


MIXES = {"zeros": (_zeros, F64_ORDERS), "nans": (_nans, F64_ORDERS), "infs": (_infs, F64_ORDERS),
         "normal": (_normal, F64_ORDERS), "i64_heavy": (_i64_heavy, I64_ORDERS)}


@functools.lru_cache(maxsize=8)
def _mix(name, n):
    return _records(MIXES[name][0](np.random.default_rng([len(name), n]), n))


def _sort(a, flags, radix=16):
    with lsb.DistributedSorter(len(a), radix_bits=radix, flags=flags) as s:
        s.upload(a)
        st = s.my_sort()
        return s.download(), st


def _check(a, order, shapes=SHAPES, radix=16):
    korder = KO.ORDERS[order]
    want = KO.reference(a, korder)
    enc = KO.order_key(a["key"], korder)
    for flags in shapes:
        got, st = _sort(a, korder | flags, radix)
        _assert_same(got, want, order, len(a), radix, flags)
        assert st.skipped == _expected_skips(enc, flags, radix), (order, len(a), radix, flags, st.skipped)


# ---- 1. orders x shapes x sizes ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("order", ORDERS)
def test_orders_bit_exact(order, n):
    _check(_records(_mixed(n, 1)), order)


# ---- 2. every pattern read as the typed key, and the special-value mixes ----------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("name", P.PATTERNS)
def test_patterns_as_typed_keys(name, order):
    _check(P.make(name, P.SUPERTILE + 1), order, shapes=[0, TL, OP, TL | OP])


@pytest.mark.parametrize("n", [P.SUPERTILE + 1, (1 << 20) + 7])
@pytest.mark.parametrize("mix,order", [(m, o) for m, (_, orders) in MIXES.items() for o in orders])
def test_special_value_mixes(mix, order, n):
    a = _mix(mix, n)
    _check(a, order)
    if mix == "zeros":  # stability across -0.0 / +0.0: both kinds of zero keep their input order among each other
        got, _ = _sort(a, KO.ORDERS[order])
        z = (got["key"] << np.uint64(1)) == 0
        assert (np.diff(got["val"][z].astype(np.int64)) > 0).all()
        assert set(got["key"][z].tolist()) == {0, 1 << 63}


# ---- 3. radix widths: the sign bit sits in a partial last digit at 11 and 13 -------------------------------------------
@pytest.mark.parametrize("radix", [1, 8, 11, 13, 16])
@pytest.mark.parametrize("order", ORDERS)
def test_radix_widths(order, radix):
    n = P.PART_TILE * 3 + 5 if radix == 1 else P.SUPERTILE + 1
    keys = _mix("i64_heavy", n)["key"] if order in I64_ORDERS else _mixed(n, 2)
    _check(_records(keys), order, shapes=[0, TL, OP, TL | OP], radix=radix)


# ---- 4. skips follow the varying bits of order_key(keys) ----------------------------------------------------------------
def test_skips_on_constant_ordered_digits():
    n = P.SUPERTILE + 1
    rng = np.random.default_rng(3)
    in_1_2 = _records((1.0 + rng.random(n)).view(np.uint64))  # exponent 0x3FF: the top 12 bits of order_key are constant
    pay = rng.integers(1, 1 << 52, n, dtype=np.uint64)
    all_nan = _records(np.uint64(0x7FF0000000000000) | pay | (rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63)))
    for a, name in ((in_1_2, "[1,2)"), (all_nan, "nan")):
        for order in F64_ORDERS:
            enc = KO.order_key(a["key"], KO.ORDERS[order])
            for radix in (8, 16):
                assert _expected_skips(enc, 0, radix) > 0, (name, radix)
                _check(a, order, radix=radix)
    # every NaN is the same key: every step is skipped and the array stays in input order
    got, st = _sort(all_nan, KO.F64)
    assert st.skipped == 8 and (got == all_nan).all()


# ---- 5. pass by pass against the oracle on order_key(keys) --------------------------------------------------------------
@pytest.mark.parametrize("flags", [0, TL], ids=["default", "two_level"])
@pytest.mark.parametrize("order", ORDERS)
def test_each_pass(order, flags):
    n = P.SUPERTILE + 1
    korder = KO.ORDERS[order]
    a = _records(_mixed(n, 4))
    cur = a.copy()
    cur["key"] = KO.order_key(a["key"], korder)  # the oracle sorts order_key as plain uint64
    with lsb.DistributedSorter(n, flags=korder | flags) as s:
        s.upload(a)
        for p in range(4):
            want, counts, starts, _ = O.one_pass(cur, n, 1, 16, p)
            assert (s.histogram(p) == counts[0]).all(), (order, flags, p)
            assert (s.starts(p) == starts[:, 0]).all(), (order, flags, p)
            s.global_shuffle(p)
            got = s.download()
            assert np.array_equal(got["val"], want["val"]), (order, flags, p)
            assert np.array_equal(got["key"], a["key"][got["val"].astype(np.int64)]), (order, flags, p)
            cur = want


# ---- 6. the exchange kernel's fused next-digit count under an order ------------------------------------------------------
@pytest.mark.parametrize("order", F64_ORDERS)
def test_fused_next_digit_count(order):
    """random bits read as doubles: every digit of order_key is wide, so each pass's exchange counts the next digit
    (as many launches as the uint64 sort of the same bits, which fuses the same way)"""
    n = (1 << 20) + 7
    a = _records(np.random.default_rng(5).integers(0, 1 << 64, n, dtype=np.uint64))
    for flags in (TL, TL | OP):
        got, st = _sort(a, KO.ORDERS[order] | flags)
        _assert_same(got, KO.reference(a, KO.ORDERS[order]), order, flags)
        _, st_u = _sort(a, flags)
        assert st.kernel_launches == st_u.kernel_launches, (order, flags)


# ---- 7. verify() -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
def test_verify_after_ordered_sort(order):
    n = (1 << 20) + 7
    a = _records(_mixed(n, 6))
    for flags in (0, TL, OP):
        with lsb.DistributedSorter(n, flags=KO.ORDERS[order] | flags) as s:
            s.upload(a)
            assert s.checksum() == O.checksum(a)
            s.my_sort()
            v = s.verify()
            assert v.order_violations == 0 and v.elements == n and list(v.checksum) == O.checksum(a), (order, flags)


def test_verify_uses_the_order():
    """negative doubles in uint64 order are descending as doubles: an f64 context must see violations"""
    n = 10000
    a = _records(np.sort((-1.0 - np.random.default_rng(8).random(n)).view(np.uint64)))
    with lsb.DistributedSorter(n, flags=KO.F64) as s:
        s.upload(a)
        v = s.verify(raise_on_failure=False)
        assert v.order_violations > 0
        with pytest.raises(lsb.LsbError):
            s.verify()
    with lsb.DistributedSorter(n) as s:
        s.upload(a)
        assert s.verify().order_violations == 0


# ---- 8. no extra kernels: the order is read inside the kernels that read digits -----------------------------------------
@pytest.mark.parametrize("order", ORDERS)
def test_no_extra_kernels(order):
    n = (1 << 20) + 7
    a = _records(np.random.default_rng(9).integers(0, 1 << 64, n, dtype=np.uint64))
    for flags in (NS, NS | OP, NS | TL, NS | TL | OP):
        _, st = _sort(a, KO.ORDERS[order] | flags)
        _, st_u = _sort(a, flags)
        assert (st.kernel_launches, st.partition_elements) == (st_u.kernel_launches, st_u.partition_elements), (order, flags)


# ---- 9. other entry points -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
def test_sort_host(order):
    n = P.SUPERTILE + 1
    a = _records(_mixed(n, 10))
    out = np.empty_like(a)
    with lsb.DistributedSorter(n, flags=KO.ORDERS[order]) as s:
        s.sort_host(a, out)
    _assert_same(out, KO.reference(a, KO.ORDERS[order]), order)


@pytest.mark.parametrize("descending", [False, True])
@pytest.mark.parametrize("dtype", [np.uint64, np.int64, np.float64])
def test_sort_pairs(dtype, descending):
    flags = KO.ORDERS[{np.uint64: "u64", np.int64: "i64", np.float64: "f64"}[dtype] + ("_desc" if descending else "")]
    for n in (0, 1, 2, 10007, P.SUPERTILE + 1):
        bits = _mixed(n, 11) if n else np.zeros(0, dtype=np.uint64)
        keys = bits.view(dtype)
        k, v = lsb.sort_pairs(keys, descending=descending)
        want = KO.argsort(bits, flags)
        assert k.dtype == dtype and v.dtype == np.int64
        assert np.array_equal(v, want), (dtype, descending, n)
        assert np.array_equal(k.view(np.uint64), bits[want]), (dtype, descending, n)  # bits unchanged: -0.0, NaN payloads
        vals = (np.arange(n, dtype=np.float64) * 0.5)
        k2, v2 = lsb.sort_pairs(keys, vals, descending=descending)
        assert v2.dtype == np.float64 and np.array_equal(v2, vals[want]) and np.array_equal(k2.view(np.uint64), bits[want])


def test_conflicting_type_flags():
    with pytest.raises(lsb.LsbError) as e:
        lsb.DistributedSorter(100, flags=KO.I64 | KO.F64)
    assert e.value.code == -1
