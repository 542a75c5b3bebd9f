"""Segmented sort without a GPU: lsb_sort_segments_device is declared and bound, the Python entry points refuse malformed
arguments before the library is reached, the bit layout compiled from csrc/lsb_segments.cuh equals hostlogic's, and a
numpy model of the algorithm (pack, key passes, retag, segment passes, unpack) equals np.lexsort((keys, segment))."""
import inspect
import os
import shutil
import subprocess

import numpy as np
import pytest

import distributed_lsb_b200 as lsb
import key_orders as KO
from distributed_lsb_b200 import hostlogic as H
from distributed_lsb_b200 import lsbsort as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- the numpy model of lsb_sort_segments_device ------------------------------------------------------------------------
def segment_ids(offsets, count):
    """segment of every input position (the search segsort_pack_kernel makes)"""
    return np.searchsorted(np.asarray(offsets, dtype=np.int64), np.arange(count), side="right") - 1


def _lsd(sort_key, words, radix, digits):
    """stable LSD passes on `digits` of sort_key(words) (the order of rows of `words` is what moves)"""
    for d in digits:
        shift = radix * d
        bits = min(radix, 64 - shift)
        dig = (sort_key(words) >> np.uint64(shift)) & np.uint64((1 << bits) - 1)
        words = words[np.argsort(dig, kind="stable")]
    return words


def model(keys, offsets, radix, flags=0, vals=None, local=False):
    """steps 2-6 of the algorithm on uint64 key bits: returns (keys_out, vals_out as uint64)"""
    keys = np.asarray(keys, dtype=np.uint64)
    n, S = len(keys), len(offsets) - 1
    idxbits, segbits, segw, passes, fits = H.segsort_layout(n, S, radix)
    assert fits
    seg = segment_ids(offsets, n).astype(np.uint64)
    rec = np.stack([keys, np.arange(n, dtype=np.uint64) | (seg << np.uint64(idxbits))], 1)       # pack
    rec = _lsd(lambda r: KO.order_key(r[:, 0], flags), rec, radix, range(H.num_passes(radix)))   # key passes
    if segbits:
        idx = rec[:, 1] & np.uint64((1 << idxbits) - 1)
        rec = np.stack([(rec[:, 1] >> np.uint64(idxbits)) | (idx << np.uint64(segw)), rec[:, 0]], 1)  # retag
        rec = _lsd(lambda r: r[:, 0], rec, radix, range(passes))                                  # segment passes
        out_k, idx, s = rec[:, 1], rec[:, 0] >> np.uint64(segw), rec[:, 0] & np.uint64((1 << segw) - 1)
    else:
        out_k, idx, s = rec[:, 0], rec[:, 1], np.zeros(n, dtype=np.uint64)
    if vals is not None:
        out_v = np.asarray(vals).view(np.uint64)[idx.astype(np.int64)]
    elif local:
        out_v = idx - np.asarray(offsets, dtype=np.int64).view(np.uint64)[s.astype(np.int64)]
    else:
        out_v = idx
    return out_k, out_v


def lexsort_reference(keys, offsets, flags=0):
    """input positions in the order of the stable sort by (segment, order_key(key))"""
    keys = np.asarray(keys, dtype=np.uint64)
    return np.lexsort((KO.order_key(keys, flags), segment_ids(offsets, len(keys))))


def ragged_offsets(rng, n, S):
    """S segments of random sizes (many empty when S is large against n) over n elements"""
    cuts = np.sort(rng.integers(0, n + 1, S - 1))
    return np.concatenate([[0], cuts, [n]]).astype(np.int64)


def _cases():
    rng = np.random.default_rng(5)
    yield "one", 100, np.array([0, 100])
    yield "rows", 96, np.arange(0, 97, 8)
    yield "len1", 50, np.arange(51)
    yield "empty_first_inside_last", 40, np.array([0, 0, 0, 10, 10, 25, 40, 40, 40])
    yield "huge_among_tiny", 300, np.array([0, 1, 2, 290, 291, 293, 300])
    for S in (255, 256, 257, 2049):
        yield f"ragged{S}", 3000, ragged_offsets(rng, 3000, S)
    yield "zero", 0, np.zeros(4, dtype=np.int64)
    yield "single", 1, np.array([0, 0, 1, 1])


@pytest.mark.parametrize("radix", [8, 11, 13, 16])
def test_model_equals_lexsort(radix):
    rng = np.random.default_rng(radix)
    for name, n, off in _cases():
        for order in ("u64", "i64_desc", "f64", "f64_desc"):
            flags = KO.ORDERS[order]
            keys = KO.special_mix(n, seed=n) if n else np.zeros(0, dtype=np.uint64)
            if n and order == "u64":
                keys = rng.integers(0, 4, n, dtype=np.uint64) << np.uint64(62)  # heavy ties: stability shows
            perm = lexsort_reference(keys, off, flags)
            k, v = model(keys, off, radix, flags)
            assert np.array_equal(k, keys[perm]) and np.array_equal(v, perm.astype(np.uint64)), (name, order, radix)
            vals = rng.standard_normal(n)
            k, v = model(keys, off, radix, flags, vals=vals)
            assert np.array_equal(v, vals.view(np.uint64)[perm]), (name, order, radix)
            k, v = model(keys, off, radix, flags, local=True)
            seg = segment_ids(off, n)
            assert np.array_equal(v.astype(np.int64), perm - off[seg[perm]]), (name, order, radix)


# ---- the bit layout: C++ header == hostlogic mirror ---------------------------------------------------------------------
PROG = r'''
#include <cstdio>
#include "lsb_segments.cuh"
int main() {  // "count num_segments radix_bits" lines on stdin -> "idxbits segbits segw passes fits" lines
  long long n, s;
  int r;
  while (scanf("%lld %lld %d", &n, &s, &r) == 3) {
    const lsb::SegsortLayout l = lsb::segsort_layout(n, s, r);
    printf("%d %d %d %d %d\n", l.idxbits, l.segbits, l.segw, l.passes, (int)l.fits);
  }
  return 0;
}
'''

LAYOUT_CASES = [(n, s, r) for n in (0, 1, 2, 3, 1 << 20, (1 << 30) + 1, 1 << 32, (1 << 40) + 3, (1 << 63) - 1)
                for s in (-1, 0, 1, 2, 255, 256, 257, 65535, 65536, 65537, 1 << 30, (1 << 30) + 1, 1 << 40)
                for r in (0, 1, 8, 11, 13, 16, 17)]


def test_layout_header_equals_hostlogic(tmp_path):
    cxx = shutil.which("g++") or shutil.which("c++")
    if cxx is None:
        pytest.skip("no C++ compiler")
    (tmp_path / "prog.cpp").write_text(PROG)
    exe = tmp_path / "prog"
    subprocess.check_call([cxx, "-std=c++17", "-D__host__=", "-D__device__=", "-I",
                           os.path.join(ROOT, "distributed-lsb_b200", "csrc"), str(tmp_path / "prog.cpp"), "-o", str(exe)])
    text = "".join(f"{n} {s} {r}\n" for n, s, r in LAYOUT_CASES)
    got = subprocess.run([str(exe)], input=text, capture_output=True, text=True, check=True).stdout.split("\n")
    for (n, s, r), line in zip(LAYOUT_CASES, got):
        want = H.segsort_layout(n, s, r)
        assert tuple(int(x) for x in line.split()) == tuple(int(x) for x in want), (n, s, r)


def test_layout_examples():
    assert H.segsort_layout(1 << 30, 256, 16) == (30, 8, 16, 1, True)       # 256 segments: one 16-bit pass, its high
    assert H.segsort_layout(1 << 30, 1, 16) == (30, 0, 0, 0, True)          # step constant; one segment: no pass
    assert H.segsort_layout(1 << 32, 1 << 32, 16) == (32, 32, 32, 2, True)  # radix 16, count <= 2^32: always fits
    assert H.segsort_layout(1 << 30, 1 << 30, 13) == (30, 30, 39, 3, False)  # 39 + 30 bits: refused
    assert H.segsort_layout(0, 5, 8) == (1, 3, 8, 1, True)
    assert not H.segsort_layout(10, 0, 16)[4]


# ---- the ABI and the Python argument checks -----------------------------------------------------------------------------
def test_declared_and_bound():
    assert "lsb_sort_segments_device" in lsb.header_symbols()
    assert "L.lsb_sort_segments_device.argtypes" in inspect.getsource(L.load_library)
    header = open(os.path.join(ROOT, "include", "lsbsort.h")).read()
    assert "#define LSB_SEG_LOCAL_INDEX 1u" in header and L.SEG_LOCAL_INDEX == 1


torch = pytest.importorskip("torch")


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"library called ({name}) before the arguments were checked")


def _sorter(here=16, flags=0, device=0):
    s = object.__new__(L.DistributedSorter)
    s._L, s._ctx = _NoLibrary(), None
    s.here, s.device, s.flags = here, device, flags
    return s


def test_sorter_rejects_bad_offsets():
    s = _sorter(here=16, flags=L.FLAG_KEY_I64)
    keys = torch.zeros(16, dtype=torch.int64)
    for off, err, what in [([0, 16], TypeError, "torch.Tensor"), (torch.tensor([0, 16], dtype=torch.int32), TypeError, "int64"),
                           (torch.tensor([0.0, 16.0]), TypeError, "int64"), (torch.zeros(2, 2, dtype=torch.int64), ValueError, "1-D"),
                           (torch.zeros(1, dtype=torch.int64), ValueError, "at least 2"),
                           (torch.zeros(8, dtype=torch.int64)[::2], ValueError, "contiguous"),
                           (torch.tensor([0, 16]), ValueError, "CUDA")]:
        with pytest.raises(err, match=what):
            s.sort_segments(keys, off)


def test_oneshot_rejects():
    i64 = lambda *shape: torch.zeros(*shape, dtype=torch.int64)  # noqa: E731
    for args, err in [((i64(16),), ValueError),                          # 1-D without offsets
                      ((i64(4, 4), i64(5)), ValueError),                 # 2-D with offsets
                      ((i64(2, 2, 4),), ValueError),                     # 3-D
                      ((i64(4, 4),), ValueError),                        # on the CPU
                      ((torch.zeros(4, 4, dtype=torch.int32),), TypeError),
                      ((torch.zeros(4, 4, dtype=torch.float32),), TypeError),
                      (([1, 2],), TypeError)]:
        with pytest.raises(err):
            lsb.sort_segments(*args)
    with pytest.raises(ValueError, match="shape"):
        lsb.sort_segments(i64(4, 4), vals=i64(4, 3))
    with pytest.raises(TypeError):
        lsb.sort_segments(i64(4, 4), vals=[0] * 16)
