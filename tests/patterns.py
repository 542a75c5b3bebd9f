"""Structured inputs for the sort's data-dependent paths (numpy, seeded, deterministic) and their reference answer.

Random keys rarely reach the paths that depend on the data: sorted and reverse-sorted input, runs of equal keys the size
of a warp row or of a kernel's tile, one key that holds most of the array, a digit that is constant except for one
element, a digit the fused next-digit count sees as wide in its sample and narrow everywhere else.  Every pattern here
is a function of (name, n) alone, so a failure can be reproduced from the test id.

The reference is numpy's stable argsort by key: it shares no code with the library or the C oracle, and it is the
answer for every radix and every pass shape.
"""
import zlib

import numpy as np

ELT = np.dtype([("key", "<u8"), ("val", "<u8")])

K = 0x8899AABBCCDDEEFF             # every byte distinct, top bit set
PART_TILE = 5632                   # partition_kernel tile (512 threads x 11)
ONEPASS_TILE = 2816                # onepass_kernel tile (256 threads x 11)
SUPERTILE = 232 * ONEPASS_TILE     # one-pass supertile at the default op_t1
SAMPLE = 65536                     # elements plan_fusion looks at
MASK64 = (1 << 64) - 1

# the odd element of "all_but_one_*": one bit away from K, chosen so that it has to move
ODD = {"first": K | (1 << 34),   # bit 34 of K is 0: larger than K, goes to the end
       "mid": K & ~(1 << 9),      # bit 9 of K is 1: smaller, goes to the front
       "last": K & ~(1 << 63)}    # smaller, goes to the front


def _rng(name, n, salt=0):
    return np.random.default_rng([zlib.crc32(name.encode()), n, salt])


def _random(rng, n):
    return rng.integers(0, 1 << 64, n, dtype=np.uint64, endpoint=False)


def _ascending(rng, n):
    # distinct, strictly increasing, spread over the whole key range (gaps < 2^64 / (n + 1) cannot overflow)
    return np.cumsum(rng.integers(1, MASK64 // (n + 1), n, dtype=np.uint64), dtype=np.uint64)


def _heavy(f):
    def gen(rng, n):
        k = _random(rng, n)
        k[rng.random(n) < f] = K
        return k
    return gen


def _all_but_one(where):
    def gen(rng, n):
        k = np.full(n, K, dtype=np.uint64)
        pos = {"first": 0, "mid": n // 2, "last": n - 1}[where]
        k[pos] = ODD[where]
        return k
    return gen


def _one_bit(bit):
    def gen(rng, n):
        base = np.uint64(K & ~(1 << bit))
        return base | (rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(bit))
    return gen


def _runs(length):
    def gen(rng, n):
        return np.repeat(_random(rng, n // length + 1), length)[:n]
    return gen


def _sawtooth(period):
    # 0, 1, .., P-1, 0, 1, ..: the same value in every 16-bit digit, so every pass of every radix sees the saw
    def gen(rng, n):
        return (np.arange(n, dtype=np.uint64) % np.uint64(period)) * np.uint64(0x0001000100010001)
    return gen


def _few(k):
    # k distinct keys that differ in every 16-bit digit, at random positions
    def gen(rng, n):
        table = np.zeros(k, dtype=np.uint64)
        for d in range(4):
            table |= rng.choice(65536, k, replace=False).astype(np.uint64) << np.uint64(16 * d)
        return table[rng.integers(0, k, n)]
    return gen


def _supertile_segments(rng, n):
    # the low byte of digit 0 is constant within each one-pass supertile and changes from one to the next: each
    # supertile is a single segment of its first step
    k = _random(rng, n)
    block = (np.arange(n, dtype=np.uint64) // np.uint64(SUPERTILE)) * np.uint64(0x9D) + np.uint64(0x31)
    return (k & ~np.uint64(0xFF)) | (block & np.uint64(0xFF))


def _lying_sample(rng, n):
    # random in the first SAMPLE elements, then one value of digit 1 (radix 16): the sample says "wide digit, fuse its
    # count into pass 0's exchange", the rest of the array sends every element to one bin
    k = _random(rng, n)
    k[SAMPLE:] = (k[SAMPLE:] & ~np.uint64(0xFFFF << 16)) | np.uint64(0x5A5A << 16)
    return k


GENERATORS = {"ascending": _ascending, "descending": lambda rng, n: _ascending(rng, n)[::-1].copy()}
GENERATORS.update({f"heavy_{f}": _heavy(f) for f in (0.5, 0.9, 0.999)})
GENERATORS.update({f"all_but_one_{w}": _all_but_one(w) for w in ("first", "mid", "last")})
GENERATORS.update({"bit63_only": _one_bit(63), "bit0_only": _one_bit(0)})
GENERATORS.update({f"runs_{L}": _runs(L) for L in (31, 32, 33, 2815, 2816, 2817, 5631, 5632, 5633)})
GENERATORS.update({f"saw_{P}": _sawtooth(P) for P in (32, 2816, 5632, 65536)})
GENERATORS.update({f"few_{k}": _few(k) for k in (2, 255, 256, 257)})
GENERATORS.update({"supertile_segments": _supertile_segments, "lying_sample": _lying_sample})

PATTERNS = sorted(GENERATORS)
GENERATORS["random"] = _random  # the unstructured baseline, for comparisons
VALS = ("index", "small", "zero")  # arange(n); random in [0, 16); all zero


def make(name, n, vals="index"):
    """the records of pattern `name` at size n; vals other than "index" repeat, so only the multiset and the
    reference (not verify(), which needs unique vals) can check them"""
    a = np.zeros(n, dtype=ELT)
    a["key"] = GENERATORS[name](_rng(name, n), n)
    if vals == "index":
        a["val"] = np.arange(n, dtype=np.uint64)
    elif vals == "small":
        a["val"] = _rng(name, n, 1).integers(0, 16, n, dtype=np.uint64)
    else:
        assert vals == "zero", vals
    return a


def reference(a):
    """the stable sort by key"""
    return a[np.argsort(a["key"], kind="stable")]


# The library's built-in values of every lsb_tune key except the partition_kernel ones (those are LIB_DEFAULT_TUNE in
# tests/conftest.py): Tuning in csrc/lsbsort.cu.  Tests that change a tunable put these back afterwards.
TUNE_DEFAULTS = {"op_cfg": 1, "op_t1": 232, "op_nx": 6, "op_lead": 3, "op_hints": 15, "op_persist": 0, "op_ctas_mgpu": 3,
                 "timeout_ms": 4000, "vparts": 16, "vramp": 130, "ex_ctas": 1, "ex_threads": 0, "ex_u": 4}


def digit(keys, shift, bits):
    return ((keys >> np.uint64(shift)) & np.uint64((1 << bits) - 1)).astype(np.int64)
