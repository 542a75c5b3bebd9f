"""The key orders of include/lsbsort.h for the tests: a numpy restatement of order_key (csrc/lsb_keyorder.cuh), used
for digit-level expectations (counts, skips, the oracle's single pass), and the reference for whole sorts: numpy's
stable argsort on the typed view of the keys, which shares no code with order_key.
"""
import numpy as np

from distributed_lsb_b200 import lsbsort as L

I64, F64, DESC = L.FLAG_KEY_I64, L.FLAG_KEY_F64, L.FLAG_DESCENDING
TOP = np.uint64(1 << 63)
ALL = np.uint64((1 << 64) - 1)
ORDERS = {"u64": 0, "u64_desc": DESC, "i64": I64, "i64_desc": I64 | DESC, "f64": F64, "f64_desc": F64 | DESC}
DTYPES = {0: np.uint64, I64: np.int64, F64: np.float64}


def order_key(keys, flags):
    """uint64 keys -> the uint64 whose ascending stable sort is the sort under `flags`"""
    k = np.array(keys, dtype=np.uint64, copy=True)
    if flags & F64:
        k[(k << np.uint64(1)) == 0] = 0                                   # -0.0 -> +0.0
        nan = (k << np.uint64(1)) > np.uint64(0x7FF << 53)
        k ^= (k.view(np.int64) >> np.int64(63)).view(np.uint64) | TOP
        k[nan] = ALL
    elif flags & I64:
        k ^= TOP
    return ~k if flags & DESC else k


def typed(keys, flags):
    return np.asarray(keys, dtype=np.uint64).view(DTYPES[flags & (I64 | F64)])


def argsort(keys, flags):
    """numpy's stable argsort of the typed view; descending: the stable ascending sort of the reversed array, reversed
    (equal keys stay in input order)"""
    x = typed(keys, flags)
    if not flags & DESC:
        return np.argsort(x, kind="stable")
    n = len(x)
    return (n - 1 - np.argsort(x[::-1], kind="stable"))[::-1]


def reference(a, flags):
    """the records of `a` in sorted order"""
    return a[argsort(a["key"], flags)]


def f64_bits(values):
    return np.asarray(values, dtype=np.float64).view(np.uint64)


# special values: +-0, +-inf, quiet and signalling NaNs of both signs with payloads, +- the smallest subnormal,
# +- the largest finite double, and the int64 extremes, 0 and -1 (as bit patterns they are also doubles and uint64s)
SPECIAL_BITS = np.array([
    0x0000000000000000, 0x8000000000000000,                      # +0.0 / int64 0, -0.0 / int64 min
    0x7FF0000000000000, 0xFFF0000000000000,                      # +inf, -inf
    0x7FF8000000000000, 0xFFF8000000000000,                      # quiet NaN, both signs
    0x7FF8000000000123, 0xFFFC0000000ABCDE,                      # quiet NaNs with payloads
    0x7FF0000000000001, 0xFFF0000000000001, 0x7FF4000000000042,  # signalling NaNs
    0x0000000000000001, 0x8000000000000001,                      # +- smallest subnormal
    0x7FEFFFFFFFFFFFFF, 0xFFEFFFFFFFFFFFFF,                      # +- largest finite
    0x3FF0000000000000, 0xBFF0000000000000,                      # +-1.0
    0x7FFFFFFFFFFFFFFF, 0xFFFFFFFFFFFFFFFF,                      # int64 max, -1 (both NaNs as doubles)
], dtype=np.uint64)


def special_mix(n, seed=0):
    """n keys drawn from SPECIAL_BITS and from standard-normal doubles, shuffled"""
    rng = np.random.default_rng(seed)
    k = np.concatenate([SPECIAL_BITS[rng.integers(0, len(SPECIAL_BITS), n - n // 2)],
                        rng.standard_normal(n // 2).view(np.uint64)])
    return k[rng.permutation(n)]
