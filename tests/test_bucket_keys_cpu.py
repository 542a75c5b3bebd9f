"""A numpy model of the 32-bit chunk keys of bucket_sort_kernel (csrc/lsb_bucket.cuh) and of the rule that sends a
chunk to the 64-bit keys: when the rule lets a chunk pass, the 32-bit order is the stable sort of its order keys, and
every chunk whose 32-bit order is not the stable sort is caught -- no GPU needed."""
import numpy as np
import pytest

U64 = np.uint64
C = 256


def chunk_keys(ordinal, low, low_bits):
    """(32-bit keys, prefix drops low bits) of one chunk: (ordinal << (24 - w) | prefix) << 8 | pos, padded to 32 * R
    with 0xFFFFFFFF"""
    n = len(ordinal)
    w = int(ordinal.max()).bit_length()
    pw = 24 - w
    drop = max(low_bits - pw, 0)
    keys = ((ordinal.astype(np.uint64) << U64(pw) | (low >> U64(drop))) << U64(8) | np.arange(n, dtype=U64))
    r = 2 if n <= 64 else 4 if n <= 128 else 8
    pad = np.full(32 * r - n, 0xFFFFFFFF, dtype=U64)
    return np.concatenate([keys, pad]), drop > 0


def model(ordinal, low, low_bits):
    """(rank -> chunk position from the 32-bit keys, falls back)"""
    keys, dropped = chunk_keys(ordinal, low, low_bits)
    assert keys.max() <= 0xFFFFFFFF
    s = np.sort(keys)  # the bitonic network; keys are distinct by pos, the padding sorts last
    n = len(ordinal)
    assert (s[n:] == 0xFFFFFFFF).all() and (s[:n] < 0xFFFFFFFF).all()
    perm = (s[:n] & U64(255)).astype(np.int64)
    full = ordinal.astype(np.uint64) << U64(low_bits) | low  # stands for the order key within the chunk
    tie = (s[1:n] >> U64(8)) == (s[:n - 1] >> U64(8))
    bad = dropped and bool((tie & (full[perm[1:]] != full[perm[:-1]])).any())
    return perm, bad


def chunk(rng, sizes, low_bits, low):
    ordinal = np.repeat(np.arange(len(sizes)), sizes)
    return ordinal, low(rng, len(ordinal), low_bits)


def uniform(rng, n, lb):
    return rng.integers(0, 1 << lb, n, dtype=U64)


CASES = {
    # every chunk falls back: the prefix sees only constant bits
    "constant_prefix": (40, [100, 90, 60], lambda r, n, lb: U64(0x3C3C3C << 16) | r.integers(0, 1 << 16, n, dtype=U64)),
    # some: a few values per bucket, apart only in the last bits
    "few_values": (40, [50, 70, 3, 1], lambda r, n, lb: r.choice(np.array([7 << 20, 7 << 20 | 1, 9 << 30], dtype=U64), n)),
    "equal_keys": (40, [200, 56], lambda r, n, lb: r.choice(np.array([5, 1 << 39], dtype=U64), n)),
    # none: k = 7, the prefix is exact
    "exact_k7": (8, [30, 30, 30, 30, 30, 30, 30, 30], uniform),
    "widest_ordinal": (8, [1] * 256, uniform),
    "exact_k6": (16, [1] * 200 + [56], uniform),
    "k2": (48, [40, 40, 40, 40, 40, 40], uniform),
    "k3": (40, [64, 64, 64, 64], uniform),
    "full_256": (40, [256], lambda r, n, lb: r.choice(np.array([0, 0, 2, 1 << 20, 9], dtype=U64), n)),
    "short": (40, [3, 2], uniform),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_rule_equals_stable_sort(name):
    lb, sizes, low = CASES[name]
    rng = np.random.default_rng(len(name))
    for _ in range(200):
        ordinal, low_part = chunk(rng, sizes, lb, low)
        perm, bad = model(ordinal, low_part, lb)
        full = ordinal.astype(np.uint64) << U64(lb) | low_part
        stable = np.argsort(full, kind="stable")
        # passing chunks are in stable order: every tie that makes the 32-bit order wrong is caught
        assert bad or (perm == stable).all()


def test_fallback_rates():
    rng = np.random.default_rng(1)
    fell = {name: 0 for name in CASES}
    for name, (lb, sizes, low) in CASES.items():
        for _ in range(50):
            fell[name] += model(*chunk(rng, sizes, lb, low), lb)[1]
    assert fell["constant_prefix"] == 50
    assert 0 < fell["few_values"] <= 50
    assert fell["equal_keys"] == 0  # equal order keys are already in pos order
    assert fell["exact_k7"] == fell["widest_ordinal"] == fell["exact_k6"] == 0


def test_padding_sorts_after_every_record():
    # the largest real key of a padded chunk: largest ordinal, prefix all ones, pos 32 * R - 2
    for n in (63, 127, 255):
        ordinal = np.zeros(n, dtype=np.int64)
        ordinal[-1] = 255 if n == 255 else 63
        keys, _ = chunk_keys(ordinal, np.full(n, (1 << 40) - 1, dtype=U64), 40)
        assert keys[:n].max() < 0xFFFFFFFF
