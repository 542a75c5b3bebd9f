"""Key columns for the lexsort tests: bit patterns of the ten key types and the reference order of a sort by several
columns -- np.lexsort over each column's dense ranks, taken from numpy's own comparison of the typed values (bfloat16
through its exact float32 widening), with every NaN one rank after all numbers, -0.0 and +0.0 one rank, and a descending
column's ranks reversed.  It shares no code with order_key / order_key_narrow (csrc/lsb_keyorder.cuh).
"""
import numpy as np

import key_orders as KO
import narrow_keys as NK

WIDE = {"uint64": np.uint64, "int64": np.int64, "float64": np.float64}
NAMES = list(WIDE) + NK.NAMES
WIDTH = {**{name: 64 for name in WIDE}, **NK.BITS}
UINT = {64: np.uint64, 32: np.uint32, 16: np.uint16}


def typed(bits, name):
    """bit patterns (numpy uint64 / uint32 / uint16) as values numpy orders like the key type"""
    if name in WIDE:
        return np.ascontiguousarray(bits, dtype=np.uint64).view(WIDE[name])
    return NK.typed(bits, name)


def ranks(bits, name, descending=False):
    """dense rank of every key among the column's distinct values (numpy's ==: NaNs one value, last; -0.0 == +0.0)"""
    x = typed(bits, name)
    if len(x) == 0:
        return np.zeros(0, dtype=np.int64)
    _, inv = np.unique(x, return_inverse=True, equal_nan=True)
    inv = inv.reshape(-1).astype(np.int64)
    return inv.max() - inv if descending else inv


def reference(columns, names, descending):
    """input indices in the order of the stable sort by (column K-1, ..., column 0): np.lexsort's convention"""
    if len(columns[0]) == 0:
        return np.zeros(0, dtype=np.int64)
    return np.lexsort([ranks(b, n, d) for b, n, d in zip(columns, names, descending)])


def special_mix(n, name, seed=0):
    """n bit patterns of the type: special values (NaNs with payloads, infinities, +-0, subnormals, extremes), uniform
    bits and normal values, shuffled"""
    if name in WIDE:
        return KO.special_mix(n, seed=seed)
    return NK.special_mix(n, name, seed=seed)


def few_values(n, name, k, seed=0):
    """n keys drawn from k distinct bit patterns of the type (with -0.0 beside +0.0 and a NaN for the floats), so that
    lower columns decide most ties"""
    rng = np.random.default_rng([seed, k, WIDTH[name]])
    pool = special_mix(max(4 * k, 64), name, seed=seed + 1)
    pool = pool[rng.choice(len(pool), k, replace=False)]
    return pool[rng.integers(0, k, n)]


def to_device(torch, bits, name):
    """numpy bit patterns -> a CUDA tensor of the key type holding the same bits"""
    if name in WIDE:
        return torch.from_numpy(np.ascontiguousarray(bits, dtype=np.uint64).view(np.int64)).cuda().view(getattr(torch, name))
    return NK.to_device(torch, bits, name)
