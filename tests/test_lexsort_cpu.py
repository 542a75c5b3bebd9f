"""Sort by several key columns without a GPU: lsb_lexsort_device is declared and bound, the rounds compiled from
csrc/lsb_lexsort.cuh equal hostlogic's, a numpy model of the algorithm (pack, one stable LSD run per round on its word,
gather pack, unpack) equals np.lexsort over dense ranks, and the Python entry points refuse malformed arguments before
the library is reached."""
import inspect
import itertools
import os
import shutil
import subprocess

import numpy as np
import pytest

import distributed_lsb_b200 as lsb
import key_orders as KO
import lexsort_ref as R
from distributed_lsb_b200 import hostlogic as H
from distributed_lsb_b200 import lsbsort as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the rounds: C++ header == hostlogic mirror ------------------------------------------------------------------------
PROG = r'''
#include <cstdio>
#include "lsb_lexsort.cuh"
int main() {  // "radix K w_0 .. w_K-1" lines on stdin -> "first ncols bits passes" per round, one line per case
  int r, k;
  while (scanf("%d %d", &r, &k) == 2) {
    int w[8];
    for (int i = 0; i < k; i++) scanf("%d", &w[i]);
    lsb::LexsortRound rounds[8];
    const int n = lsb::lexsort_rounds(w, k, r, rounds);
    for (int i = 0; i < n; i++) printf("%d %d %d %d ", rounds[i].first, rounds[i].ncols, rounds[i].bits, rounds[i].passes);
    printf("\n");
  }
  return 0;
}
'''

ROUND_CASES = ([(r, ws) for k in range(1, 7) for ws in itertools.product((16, 32, 64), repeat=k) for r in range(1, 17)]
               + [(0, (64,)), (17, (32,)), (16, (8,)), (16, (32, 24)), (16, ())])


def test_rounds_header_equals_hostlogic(tmp_path):
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    (tmp_path / "prog.cpp").write_text(PROG)
    exe = tmp_path / "prog"
    subprocess.check_call([cxx, "-std=c++17", "-D__host__=", "-D__device__=", "-I",
                           os.path.join(ROOT, "distributed-lsb_b200", "csrc"), str(tmp_path / "prog.cpp"), "-o", str(exe)])
    text = "".join(f"{r} {len(ws)} {' '.join(map(str, ws))}\n" for r, ws in ROUND_CASES)
    got = subprocess.run([str(exe)], input=text, capture_output=True, text=True, check=True).stdout.split("\n")
    for (r, ws), line in zip(ROUND_CASES, got):
        want = [x for rnd in H.lexsort_rounds(list(ws), r) for x in rnd]
        assert [int(x) for x in line.split()] == want, (r, ws)


def test_rounds_examples():
    assert H.lexsort_rounds([32, 32], 16) == [(0, 2, 64, 4)]                    # (int32, float32): one 64-bit sort
    assert H.lexsort_rounds([64, 16], 16) == [(0, 1, 64, 4), (1, 1, 16, 1)]
    assert H.lexsort_rounds([16] * 5, 16) == [(0, 4, 64, 4), (4, 1, 16, 1)]     # at most 4 columns, 64 bits, a round
    assert H.lexsort_rounds([64], 13) == [(0, 1, 64, 5)]
    assert H.lexsort_rounds([16, 16, 32], 16) == [(0, 3, 64, 4)]                # (bfloat16, int16, int32)
    assert H.lexsort_rounds([64, 64, 64], 16) == [(0, 1, 64, 4), (1, 1, 64, 4), (2, 1, 64, 4)]
    assert H.lexsort_rounds([32, 64, 32], 11) == [(0, 1, 32, 3), (1, 1, 64, 6), (2, 1, 32, 3)]
    assert H.lexsort_rounds([16, 32], 13) == [(0, 2, 48, 4)]
    assert H.lexsort_rounds([], 16) == [] and H.lexsort_rounds([32], 0) == [] and H.lexsort_rounds([8], 16) == []


def test_rounds_are_fewest():
    """greedy packing of consecutive columns: no split of the widths into runs of <= 64 bits and <= 4 columns has fewer"""
    for k in range(1, 7):
        for ws in itertools.product((16, 32, 64), repeat=k):
            best = {0: 0}
            for end in range(1, k + 1):
                best[end] = min(best[s] + 1 for s in range(max(0, end - 4), end) if sum(ws[s:end]) <= 64)
            assert len(H.lexsort_rounds(list(ws), 16)) == best[k], ws


# ---- the numpy model of lsb_lexsort_device ------------------------------------------------------------------------------
def order_narrow(bits, name, descending):
    """order_key_narrow restated: the W-bit order key as uint64"""
    w = R.WIDTH[name]
    k = np.asarray(bits).astype(np.uint64)
    allb, sign = np.uint64((1 << w) - 1), np.uint64(1 << (w - 1))
    if name.startswith("int"):
        k = k ^ sign
    elif name.startswith("float") or name == "bfloat16":
        inf = {"float32": 0x7F800000, "float16": 0x7C00, "bfloat16": 0x7F80}[name]
        mag = (k << np.uint64(1)) & allb
        k = np.where(mag == 0, np.uint64(0), k)
        k = np.where(mag > np.uint64((inf << 1) & ((1 << w) - 1)), allb, k ^ np.where(k & sign, allb, sign))
    return ~k & allb if descending else k


def order(bits, name, descending):
    if name in R.WIDE:
        return KO.order_key(bits, {"uint64": 0, "int64": KO.I64, "float64": KO.F64}[name] | (KO.DESC if descending else 0))
    return order_narrow(bits, name, descending)


def model(columns, names, descending, radix, vals=None):
    """the rounds on the host: pack (index in the val word), the stable digit passes of each round, the gather pack of
    the next round at the indices the records carry, the unpack"""
    n = len(columns[0])
    idx = np.arange(n, dtype=np.int64)
    for r, (first, ncols, bits, passes) in enumerate(H.lexsort_rounds([R.WIDTH[x] for x in names], radix)):
        word, shift = np.zeros(n, dtype=np.uint64), 0
        for c in range(first, first + ncols):
            word |= order(np.asarray(columns[c])[idx], names[c], descending[c]) << np.uint64(shift)
            shift += R.WIDTH[names[c]]
        assert shift == bits
        for d in range(passes):
            lo = radix * d
            dig = (word >> np.uint64(lo)) & np.uint64((1 << min(radix, bits - lo)) - 1)
            p = np.argsort(dig, kind="stable")
            word, idx = word[p], idx[p]
    return idx if vals is None else np.asarray(vals)[idx]


MIXES = [("int32", "float32"), ("bfloat16", "int16", "int32"), ("int64", "int64"), ("int64", "int64", "int64"),
         ("float64", "bfloat16", "uint16", "float16", "uint32", "int64"), ("float16",) * 5, ("uint64",),
         ("float32", "uint64", "int16", "float64")]


@pytest.mark.parametrize("radix", [8, 11, 13, 16])
@pytest.mark.parametrize("mix", range(len(MIXES)))
def test_model_equals_lexsort(mix, radix):
    names = MIXES[mix]
    rng = np.random.default_rng([mix, radix])
    for n in (0, 1, 2, 777):
        for trial in range(3):
            cols = [R.few_values(n, name, k=3 + trial, seed=c) if c < len(names) - 1 or trial else R.special_mix(n, name, c)
                    for c, name in enumerate(names)]
            desc = [bool(x) for x in rng.integers(0, 2, len(names))]
            want = R.reference(cols, names, desc)
            assert np.array_equal(model(cols, names, desc, radix), want), (names, n, desc)
            vals = rng.standard_normal(n)
            assert np.array_equal(model(cols, names, desc, radix, vals).view(np.uint64), vals.view(np.uint64)[want])


def test_reference_rules():
    """the reference's own rules on a hand-made case: NaNs last (first descending), -0.0 == +0.0, ties by the next key"""
    f = np.array([1.0, np.nan, -0.0, 0.0, -np.nan, 1.0]).view(np.uint64)
    s = np.array([5, 4, 3, 2, 1, 0], dtype=np.uint64)
    assert list(R.reference([s, f], ["uint64", "float64"], [False, False])) == [3, 2, 5, 0, 4, 1]
    assert list(R.reference([s, f], ["uint64", "float64"], [False, True])) == [4, 1, 5, 0, 3, 2]
    assert list(R.reference([s, f], ["uint64", "float64"], [True, False])) == [2, 3, 0, 5, 1, 4]


# ---- the ABI and the Python argument checks -----------------------------------------------------------------------------
def test_declared_and_bound():
    assert "lsb_lexsort_device" in lsb.header_symbols()
    assert "L.lsb_lexsort_device.argtypes" in inspect.getsource(L.load_library)
    assert [f[0] for f in L.KeyColumn._fields_] == ["keys", "key_type", "flags"]
    header = open(os.path.join(ROOT, "include", "lsbsort.h")).read()
    assert "typedef struct lsb_key_column {" in header and "lexsort" in lsb.__dict__


torch = pytest.importorskip("torch")


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"library called ({name}) before the arguments were checked")


def _sorter(here=16, flags=0, device=0):
    s = object.__new__(L.DistributedSorter)
    s._L, s._ctx = _NoLibrary(), None
    s.here, s.device, s.flags = here, device, flags
    return s


def test_lexsort_device_rejects():
    s = _sorter(here=16)
    z = lambda dtype, *shape: torch.zeros(*(shape or (16,)), dtype=dtype)  # noqa: E731
    for cols, err, what in [(z(torch.int64, 2, 16), TypeError, "list or tuple"), ([], ValueError, "empty"),
                            ((z(torch.int64).numpy(),), TypeError, "torch.Tensor"), ([z(torch.int8)], TypeError, "int8"),
                            ([z(torch.bool)], TypeError, "bool"), ([z(torch.int64, 4, 4)], ValueError, "1-D"),
                            ([z(torch.float32, 32)[::2]], ValueError, "contiguous"), ([z(torch.int16, 15)], ValueError, "elements"),
                            ([z(torch.float64), z(torch.bfloat16)], ValueError, "CUDA")]:
        with pytest.raises(err, match=what):
            s.lexsort_device(cols)
    with pytest.raises(ValueError, match=r"columns\[0\] has 8 elements"):
        s.lexsort_device((z(torch.int32, 8), z(torch.int64)))


def test_lexsort_device_rejects_descending_and_vals():
    s = _sorter(here=16)
    z = lambda dtype, n=16: torch.zeros(n, dtype=dtype)  # noqa: E731
    for desc, err in [("yes", TypeError), (1, TypeError), ([True], ValueError), ([True, 0], TypeError), (None, TypeError)]:
        with pytest.raises(err):
            L._check_descending(desc, 2)
    assert L._check_descending(True, 3) == [True] * 3 and L._check_descending((False, True), 2) == [False, True]
    for vals, err in [(z(torch.int32), TypeError), (z(torch.int64, 15), ValueError), ([0] * 16, TypeError)]:
        with pytest.raises(err):
            L._check_vector(torch, vals, "vals", 16)


def test_oneshot_rejects():
    i64 = lambda *shape: torch.zeros(*shape, dtype=torch.int64)  # noqa: E731
    for args, kw, err in [(([],), {}, ValueError),                              # no keys
                          ((i64(0, 5),), {}, ValueError),                       # a 2-D tensor of no rows
                          ((i64(5),), {}, ValueError),                          # 1-D tensor
                          ((i64(2, 2, 4),), {}, ValueError),                    # 3-D
                          ((5,), {}, TypeError),
                          (([[1, 2, 3, 4], i64(4)],), {}, TypeError),
                          (([torch.zeros(4, dtype=torch.int8)],), {}, TypeError),
                          (([i64(4)],), {}, ValueError),                        # on the CPU
                          (([i64(4)],), {"descending": [True, False]}, ValueError)]:
        with pytest.raises(err):
            lsb.lexsort(*args, **kw)
