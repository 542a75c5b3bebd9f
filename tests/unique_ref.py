"""The reference of lsb_unique_device, unique and unique_consecutive: groups of equal elements built from each column's
dense ranks (lexsort_ref.ranks: numpy's own comparison of the typed values, all NaNs one value, -0.0 == +0.0), never
from order_key.  Sorted mode takes the stable lexsort permutation of the rank tuples and starts a group wherever the
tuple changes; consecutive mode compares adjacent tuples in input order.
"""
import numpy as np

import lexsort_ref as LR


def reference(columns, names, descending=None, consecutive=False):
    """(index, inverse, counts) as int64 arrays for bit-pattern columns of types `names`, columns[0] the least
    significant: index[r] the first input position of group r, inverse[j] the group of position j, counts[r] its size"""
    n = len(columns[0])
    if n == 0:
        return (np.zeros(0, dtype=np.int64),) * 3
    descending = descending or [False] * len(columns)
    ranks = np.stack([LR.ranks(b, x, d) for b, x, d in zip(columns, names, descending)])
    order = np.arange(n) if consecutive else np.lexsort(ranks)
    r = ranks[:, order]
    head = np.ones(n, dtype=bool)
    head[1:] = (r[:, 1:] != r[:, :-1]).any(axis=0)
    inverse = np.empty(n, dtype=np.int64)
    inverse[order] = np.cumsum(head) - 1
    starts = np.flatnonzero(head)
    return order[starts].astype(np.int64), inverse, np.diff(np.append(starts, n)).astype(np.int64)
