"""CPU checks of tests/patterns.py: each pattern is what its name says, and its numpy reference (the stable argsort that
tests/test_gpu_patterns.py compares the GPU with) equals the C oracle's merge sort and its radix sort."""
import numpy as np
import pytest

import patterns as P
from oracle import oracle as O


def _same(x, y):
    return np.array_equal(x.view(np.uint64), y.view(np.uint64))


@pytest.mark.parametrize("name", P.PATTERNS)
def test_reference_matches_oracle(name):
    for n in (P.PART_TILE + 1, 70001):
        for vals in P.VALS:
            a = P.make(name, n, vals)
            assert _same(a, P.make(name, n, vals))  # deterministic
            want = P.reference(a)
            assert _same(O.stable_sort(a, n), want), (n, vals)
            for radix in (16, 11):
                assert _same(O.sort(a, n, 1, radix), want), (n, vals, radix)
            assert O.checksum(want) == O.checksum(a)


def test_patterns_are_what_they_say():
    n = (1 << 20) + 7
    keys = {name: P.make(name, n)["key"] for name in P.PATTERNS}
    K = np.uint64(P.K)
    asc = keys["ascending"]
    desc = keys["descending"]
    assert (asc[1:] > asc[:-1]).all() and (desc[1:] < desc[:-1]).all()
    assert asc[-1] > np.uint64(1 << 62) and desc[0] > np.uint64(1 << 62)  # spread over the key range: every digit lives
    for f in (0.5, 0.9, 0.999):
        assert abs((keys[f"heavy_{f}"] == K).mean() - f) < 0.005
    for where, pos in (("first", 0), ("mid", n // 2), ("last", n - 1)):
        k = keys[f"all_but_one_{where}"]
        odd = np.flatnonzero(k != K)
        assert odd.tolist() == [pos]
        diff = int(k[pos] ^ K)
        assert bin(diff).count("1") == 1  # one bit: one digit of any radix
        assert (P.reference(P.make(f"all_but_one_{where}", n))["key"] != k).any()  # the odd element has to move
    for bit in (63, 0):
        k = keys[f"bit{bit}_only"]
        assert set(np.unique(k ^ k[0]).tolist()) == {0, 1 << bit}
    for L in (31, 32, 33, 2815, 2816, 2817, 5631, 5632, 5633):
        k = keys[f"runs_{L}"]
        starts = np.flatnonzero(np.diff(k)) + 1
        assert (np.diff(starts) == L).all() and starts[0] == L
    for period in (32, 2816, 5632, 65536):
        k = keys[f"saw_{period}"]
        assert (k[:period] == np.arange(period, dtype=np.uint64) * np.uint64(0x0001000100010001)).all()
        assert (k[period:2 * period] == k[:period]).all()
    for k_ in (2, 255, 256, 257):
        u = np.unique(keys[f"few_{k_}"])
        assert len(u) == k_
        for d in range(4):
            assert len(np.unique(P.digit(u, 16 * d, 16))) == k_  # distinct in every 16-bit digit
    k = keys["supertile_segments"]
    low = P.digit(k, 0, 8)
    blocks = [low[i:i + P.SUPERTILE] for i in range(0, n, P.SUPERTILE)]
    assert len(blocks) == 2 and all((b == b[0]).all() for b in blocks) and blocks[0][0] != blocks[1][0]
    k = keys["lying_sample"]
    d1 = P.digit(k, 16, 16)
    assert len(np.unique(d1[:P.SAMPLE])) >= 2048  # what plan_fusion needs to fuse pass 1's count into pass 0
    assert (d1[P.SAMPLE:] == d1[-1]).all()
    for vals, check in (("small", lambda v: v.max() < 16 and len(np.unique(v)) == 16), ("zero", lambda v: (v == 0).all())):
        assert check(P.make("runs_32", n, vals)["val"])
