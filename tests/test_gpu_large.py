"""Sorts past 2^31 elements and segmented sorts whose packed word fills all 64 bits -- needs a B200 with ~150 GiB free.

Past 2^31 the input index of every record needs 32 bits, one bin can hold more than 2^31 elements and local indices
exceed int32.  A numpy reference of 2^31 keys would need tens of GiB of host memory and minutes per case, and verify()
is the library checking itself, so these cases are checked by tests/sort_check.py: plain torch on the GPU, O(n), no
code shared with the library, and complete (an output that passes it is exactly the stable sort).  It is held against
numpy here at 2^20 and at the smallest 64-bit layout, and on the CPU in test_sort_check_cpu.py.

The library allocates its context with cudaMalloc, outside torch's caching allocator, so every test first returns
torch's cached memory and skips, naming the bytes it needs, when the shared GPU has less free.
"""
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import sort_check as C  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from test_segments_cpu import segment_ids  # noqa: E402

TL, OP = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS
ERR_ARG = -1
GiB = 1 << 30

BIG = (1 << 31) + (1 << 20) + 7              # n - 1 >= 2^31: 32-bit indices
LAYOUT_64 = [(13, (1 << 24) + 13, (1 << 26) + 1),  # (radix, n, S): segw + idxbits == 64
             (12, (1 << 27) + 5, (1 << 24) + 1),
             (11, (1 << 30) + 7, (1 << 22) + 1)]
BIG_SEGMENTS, BIG_SEGMENTS_GATHER = (1 << 20) + 1, 65537  # at BIG and radix 16: 32 + 32 bits
LONG_SEGMENT = (1 << 31) + 17
REFUSED_RADIX, REFUSED_SEGMENTS = 11, (1 << 22) + 1       # at BIG: 33 + 32 = 65 bits, refused
ROWS, WIDTH = (1 << 16) + 1, (1 << 15) + 1                # 2-D form: 2^31 + 2^16 + 2^15 + 1 elements


def _need(n, arrays, nseg=0):
    """bytes a case allocates: the context's two record buffers (32 B/element), `arrays` key / value arrays of 8 B, the
    offsets, the checker's bool[n] and its chunk temporaries"""
    return 32 * n + 8 * arrays * n + 8 * (nseg + 1) + n + 12 * 8 * C.CHUNK


def _room(what, need):
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"{what} needs {need / GiB:.1f} GiB of device memory, {free / GiB:.1f} GiB free")


def _check(keys_in, keys_out, idx, korder, offsets=None):
    msg = C.check_sort(keys_in, keys_out, idx, korder, offsets)
    assert msg is None, "\n" + msg


# ---- 1. the checker agrees with numpy on the GPU ----------------------------------------------------------------------------
def test_checker_agrees_with_numpy():
    from test_gpu_segments import _reference
    n = (1 << 20) + 13
    bits = KO.special_mix(n, seed=21)
    keys = torch.from_numpy(bits.view(np.int64)).cuda().view(torch.float64)
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64 | KO.DESC) as s:
        k, v, _ = s.sort_device(keys)
    _check(keys, k, v, KO.F64 | KO.DESC)
    perm = KO.argsort(bits, KO.F64 | KO.DESC)
    assert np.array_equal(k.view(torch.int64).cpu().numpy(), bits[perm].view(np.int64))
    assert np.array_equal(v.cpu().numpy(), perm)
    bad = v.clone()
    j = int(np.flatnonzero(bits[perm][:-1] == bits[perm][1:])[0])  # equal neighbours: swapping them breaks stability
    bad[j], bad[j + 1] = v[j + 1], v[j]
    assert C.check_sort(keys, k, bad, KO.F64 | KO.DESC).startswith("check 4")

    off = C.ragged_offsets(n, 1000, "cuda", seed=22)
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64) as s:
        k, v, _ = s.sort_segments(keys, off)
        kl, vl, _ = s.sort_segments(keys, off, local_index=True)
    _check(keys, k, v, KO.F64, off)
    _check(keys, kl, C.LocalIndex(vl, off), KO.F64, off)
    perm = _reference(bits, off.cpu().numpy(), KO.F64)
    assert np.array_equal(k.view(torch.int64).cpu().numpy(), bits[perm].view(np.int64))
    assert np.array_equal(v.cpu().numpy(), perm)
    assert C.check_sort(keys, k, v, KO.F64) is not None  # the segmented output is not the sort of the whole array


# ---- 2. segment layouts of exactly 64 bits --------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [0, OP])
@pytest.mark.parametrize("radix,n,S", LAYOUT_64)
def test_segments_64_bit_layout(radix, n, S, shape):
    from test_gpu_patterns import _expected_skips
    idxbits, segbits, segw, passes, fits = H.segsort_layout(n, S, radix)
    assert fits and segw + idxbits == 64 and n - 1 >= 1 << (idxbits - 1)
    _room(f"n={n} S={S}", _need(n, 4, S))
    korder = KO.F64 if radix != 12 else 0
    keys = (C.special_doubles(n, "cuda", seed=radix) if korder else C.heavy_hitter_keys(n, "cuda", seed=radix))
    keys = keys.view(torch.float64 if korder else torch.uint64)
    off = C.ragged_offsets(n, S, "cuda", seed=radix)
    vals = C.gather_vals(n, "cuda", torch.float64)
    keys_out = torch.empty_like(keys)
    vals_out = torch.empty(n, dtype=torch.int64, device="cuda")
    small = n < 1 << 25
    if small:
        bits = keys.view(torch.int64).cpu().numpy().view(np.uint64)
        offn = off.cpu().numpy()
        seg = segment_ids(offn, n)
        perm = np.lexsort((KO.order_key(bits, korder), seg))
    with lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=korder | shape) as s:
        for what in ("global", "local", "gather"):
            _, _, st = s.sort_segments(keys, off, vals if what == "gather" else None, keys_out, vals_out,
                                       local_index=what == "local")
            assert st.elements == n and st.passes == H.num_passes(radix) + passes, (what, st.passes)
            idx = {"global": vals_out, "local": C.LocalIndex(vals_out, off), "gather": C.GatheredVals(vals_out)}[what]
            _check(keys, keys_out, idx, korder, off)
            if small:
                assert np.array_equal(keys_out.view(torch.int64).cpu().numpy(), bits[perm].view(np.int64))
                got = vals_out.cpu().numpy()
                want = {"global": perm, "local": perm - offn[seg[perm]],
                        "gather": vals.view(torch.int64).cpu().numpy()[perm]}[what]
                assert np.array_equal(got, want), what
                words = seg.astype(np.uint64) | (np.arange(n, dtype=np.uint64) << np.uint64(segw))  # retagged keys
                assert st.skipped == (_expected_skips(KO.order_key(bits, korder), shape, radix)
                                      + _expected_skips(words, shape, radix, passes=range(passes))), what


# ---- 3. sort_device past 2^31 --------------------------------------------------------------------------------------------
# (name, sorter flags, radix, [(key maker, vals gathered)]); one sorter and one set of tensors per configuration
DEVICE_CONFIGS = [
    ("u64", 0, 16, [("uniform", False), ("uniform", True), ("heavy", False)]),
    ("u64_one_pass", OP, 16, [("uniform", False), ("heavy", False)]),
    ("u64_two_level", TL, 16, [("uniform", False), ("heavy", False)]),
    ("u64_two_level_one_pass", TL | OP, 16, [("uniform", False), ("heavy", False)]),
    ("f64", KO.F64, 16, [("special", False)]),
    ("f64_one_pass", KO.F64 | OP, 16, [("special", False)]),
    ("f64_desc", KO.F64 | KO.DESC, 16, [("special", False)]),
    ("f64_desc_one_pass", KO.F64 | KO.DESC | OP, 16, [("special", False)]),
    ("i64_desc", KO.I64 | KO.DESC, 16, [("heavy", False)]),
    ("i64_desc_one_pass", KO.I64 | KO.DESC | OP, 16, [("heavy", False)]),
    ("u64_radix8", 0, 8, [("uniform", False)]),
    ("u64_radix13", 0, 13, [("uniform", False)]),
]
MAKERS = {"uniform": C.uniform_keys, "heavy": C.heavy_hitter_keys, "special": C.special_doubles}
KEY_DTYPE = {0: torch.uint64, KO.I64: torch.int64, KO.F64: torch.float64}
VERIFY_AT = (1 << 31) + 12345


@pytest.mark.parametrize("name,flags,radix,cases", DEVICE_CONFIGS, ids=[c[0] for c in DEVICE_CONFIGS])
def test_sort_device_past_2p31(name, flags, radix, cases):
    n = BIG
    korder = flags & (KO.I64 | KO.F64 | KO.DESC)
    gathered = any(g for _, g in cases)
    _room(name, _need(n, 4 if gathered else 3))
    dtype = KEY_DTYPE[korder & (KO.I64 | KO.F64)]
    keys = torch.empty(n, dtype=dtype, device="cuda")
    keys_out = torch.empty_like(keys)
    vals_out = torch.empty(n, dtype=torch.int64, device="cuda")
    with lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=flags) as s:
        for seed, (maker, gather) in enumerate(cases):
            MAKERS[maker](n, "cuda", seed=seed, out=keys)
            if maker == "heavy":
                assert int((keys.view(torch.int64) == C.HOT_KEY).sum()) > 1 << 31  # one bin of every pass > 2^31
            vals = C.gather_vals(n, "cuda") if gather else None
            _, _, st = s.sort_device(keys, vals, keys_out, vals_out)
            assert st.elements == n and st.passes == H.num_passes(radix), (maker, st.elements, st.passes)
            _check(keys, keys_out, C.GatheredVals(vals_out) if gather else vals_out, korder)
            del vals
            if name == "u64" and maker == "heavy":  # the records the sort left are what verify() reads
                _verify_past_2p31(s, n)


def _verify_past_2p31(s, n):
    """verify() passes; two adjacent records past 2^31 swapped make exactly one violation; restored, it passes again"""
    v = s.verify()
    assert v.order_violations == 0 and v.elements == n
    rec = s.download(VERIFY_AT, 2)
    assert (rec["key"] == np.int64(C.HOT_KEY).view(np.uint64)).all() and rec["val"][0] < rec["val"][1]  # a tie
    s.upload(rec[::-1].copy(), VERIFY_AT)
    v = s.verify(raise_on_failure=False)
    assert v.order_violations == 1 and v.elements == n
    s.upload(rec, VERIFY_AT)
    v = s.verify()
    assert v.order_violations == 0 and v.elements == n


# ---- 4. the segmented sort past 2^31 ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [0, OP])
def test_segments_past_2p31(shape):
    n = BIG
    korder = KO.F64 if shape == 0 else 0
    _room(f"segments shape={shape}", _need(n, 4, BIG_SEGMENTS))
    keys = (C.special_doubles(n, "cuda", seed=31) if korder else C.heavy_hitter_keys(n, "cuda", seed=31))
    keys = keys.view(torch.float64 if korder else torch.uint64)
    keys_out = torch.empty_like(keys)
    vals_out = torch.empty(n, dtype=torch.int64, device="cuda")
    off = C.ragged_offsets(n, BIG_SEGMENTS, "cuda", seed=32, long_segment=LONG_SEGMENT)
    sizes = off[1:] - off[:-1]
    assert int(sizes.max()) >= LONG_SEGMENT and int(sizes[0]) == 0 and int(sizes[-1]) == 0 and int((sizes == 0).sum()) > 1000
    with lsb.DistributedSorter(n, ranks=1, flags=korder | shape) as s:
        for local in (True, False):  # local first: 32-bit positions inside the long segment
            _, _, st = s.sort_segments(keys, off, None, keys_out, vals_out, local_index=local)
            assert st.elements == n and st.passes == H.num_passes(16) + H.segsort_layout(n, BIG_SEGMENTS, 16)[3]
            _check(keys, keys_out, C.LocalIndex(vals_out, off) if local else vals_out, korder, off)
            assert int(vals_out.max()) >= 1 << 31  # local too: positions in the long segment exceed int32
        off = C.ragged_offsets(n, BIG_SEGMENTS_GATHER, "cuda", seed=33)
        vals = C.gather_vals(n, "cuda", torch.float64)
        _, _, st = s.sort_segments(keys, off, vals, keys_out, vals_out)
        assert st.elements == n and st.passes == H.num_passes(16) + H.segsort_layout(n, BIG_SEGMENTS_GATHER, 16)[3]
        _check(keys, keys_out, C.GatheredVals(vals_out), korder, off)
        del vals
    if shape:
        return
    # radix 11: 33 bits of segment id + 32 of index do not fit one word -- refused, the outputs untouched
    off = C.ragged_offsets(n, REFUSED_SEGMENTS, "cuda", seed=34)
    keys_out.view(torch.int64).fill_(0x0BADC0DE)
    vals_out.fill_(-7)
    with lsb.DistributedSorter(n, ranks=1, radix_bits=REFUSED_RADIX, flags=korder) as s:
        with pytest.raises(lsb.LsbError) as e:
            s.sort_segments(keys, off, None, keys_out, vals_out)
        assert e.value.code == ERR_ARG and "65 bits" in str(e.value)
    assert bool((keys_out.view(torch.int64) == 0x0BADC0DE).all()) and bool((vals_out == -7).all())


@pytest.mark.parametrize("shape", [0, OP])
def test_rows_past_2p31(shape):
    n = ROWS * WIDTH
    _room(f"{ROWS} rows of {WIDTH}", _need(n, 3, ROWS))
    x = (C.uniform_keys(n, "cuda", seed=41) >> 48).view(ROWS, WIDTH)  # int64 in [-2^15, 2^15): ties in every row
    off = torch.arange(ROWS + 1, dtype=torch.int64, device="cuda") * WIDTH
    if shape == 0:
        k, i = lsb.sort_segments(x)
    else:  # what the one-shot form does, at the one-pass shape
        with lsb.DistributedSorter(n, ranks=1, flags=KO.I64 | shape) as s:
            k, i, st = s.sort_segments(x.view(-1), off, local_index=True)
            assert st.elements == n
        k, i = k.view(ROWS, WIDTH), i.view(ROWS, WIDTH)
    assert k.shape == x.shape and i.dtype == torch.int64
    _check(x.view(-1), k.view(-1), C.LocalIndex(i.view(-1), off), KO.I64, off)
    across = (1 << 31) // WIDTH  # the row holding element 2^31
    rows = torch.tensor([0, 1, across, across + 1, ROWS // 2, ROWS - 1], device="cuda")
    tk, ti = torch.sort(x[rows], dim=-1, stable=True)
    assert torch.equal(k[rows], tk) and torch.equal(i[rows], ti)
