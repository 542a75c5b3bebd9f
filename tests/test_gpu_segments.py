"""Segmented sort on the device: lsb_sort_segments_device, DistributedSorter.sort_segments and sort_segments -- needs a
B200.

The reference is np.lexsort((order_key(keys), segment)) (tests/key_orders.py), compared bit for bit: keys through
their uint64 bits (NaN payloads and -0.0 count), values exactly.  The 2-D form is also compared with
torch.sort(dim=-1, stable=True).
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import distributed_lsb_b200 as lsb  # noqa: E402
import key_orders as KO  # noqa: E402
import patterns as P  # noqa: E402
from distributed_lsb_b200 import hostlogic as H  # noqa: E402
from distributed_lsb_b200 import lsbsort as L  # noqa: E402
from test_gpu_device_sort import _bits, _dev, _dtype  # noqa: E402
from test_gpu_patterns import _expected_skips  # noqa: E402
from test_segments_cpu import ragged_offsets, segment_ids  # noqa: E402

TL, OP, NS = L.FLAG_TWO_LEVEL, L.FLAG_ONE_PASS, L.FLAG_NO_SKIP
SHAPES = [0, OP, TL]
SIZES = [0, 1, 31, 33, 3 * P.PART_TILE + 7, (1 << 20) + 13, 1 << 24]
ERR_ARG = -1


# ---- segmentations: offsets of S + 1 int64 over n elements --------------------------------------------------------------
def _one(rng, n):
    return np.array([0, n])


def _rows(rng, n):  # equal rows (the last one shorter when the length does not divide n)
    length = max(1, n // 64)
    return np.append(np.arange(0, n, length), n) if n else np.array([0, 0])


def _ragged(rng, n):
    return ragged_offsets(rng, n, int(rng.integers(2, 2000)))


def _empties(rng, n):  # empty segments first, inside and last
    inner = ragged_offsets(rng, n, 50)
    inner = np.insert(inner, 25, [inner[25]] * 5)
    return np.concatenate([[0, 0, 0], inner, [n, n]])


def _len1(rng, n):
    return np.arange(n + 1) if n else np.array([0, 0])


def _huge_among_tiny(rng, n):
    if n < 40:
        return np.array([0, n])
    tiny = np.arange(0, 21)
    return np.concatenate([tiny, [n - 10], np.arange(n - 9, n + 1)])


def _count(S):
    return lambda rng, n: ragged_offsets(rng, n, S)


SEGMENTATIONS = {"one": _one, "rows": _rows, "ragged": _ragged, "empties": _empties, "len1": _len1,
                 "huge_among_tiny": _huge_among_tiny, **{f"S{S}": _count(S) for S in (255, 256, 257, 65535, 65536, 65537)}}


def _offsets(name, n, seed=0):
    off = np.asarray(SEGMENTATIONS[name](np.random.default_rng(seed), n), dtype=np.int64)
    assert off[0] == 0 and off[-1] == n and (np.diff(off) >= 0).all()
    return off


def _reference(bits, off, korder):
    return np.lexsort((KO.order_key(bits, korder), segment_ids(off, len(bits))))


def _check(bits, off, korder, flags=0, radix=16, vals=None, local=False, sorter=None, perm=None):
    """sort `bits` (read as the order's dtype) in the segments `off` through sort_segments and compare with lexsort"""
    n = len(bits)
    kt = _dev(bits, _dtype(korder))
    ot = torch.from_numpy(off).cuda()
    s = sorter or lsb.DistributedSorter(n, ranks=1, radix_bits=radix, flags=korder | flags)
    try:
        k, v, st = s.sort_segments(kt, ot, vals, local_index=local)
        perm = _reference(bits, off, korder) if perm is None else perm
        assert np.array_equal(_bits(k), bits[perm]), (korder, flags, radix, n, len(off) - 1)
        if vals is not None:
            want = vals.view(torch.int64).cpu().numpy()[perm]
        elif local:
            want = perm - off[segment_ids(off, n)[perm]]
        else:
            want = perm
        assert np.array_equal(v.view(torch.int64).cpu().numpy(), want), (korder, flags, radix, n, len(off) - 1)
        return st, perm
    finally:
        if sorter is None:
            s.close()


# ---- 1. every key order x pass shape x size, the segmentations in turn ---------------------------------------------------
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("order", sorted(KO.ORDERS))
def test_orders_shapes_sizes(order, shape, n):
    korder = KO.ORDERS[order]
    names = sorted(SEGMENTATIONS)
    name = names[(SIZES.index(n) * 7 + sorted(KO.ORDERS).index(order) * 3 + SHAPES.index(shape)) % len(names)]
    off = _offsets(name, n, seed=n)
    bits = KO.special_mix(n, seed=n + 1) if n else np.zeros(0, dtype=np.uint64)
    with lsb.DistributedSorter(n, ranks=1, flags=korder | shape) as s:
        st, perm = _check(bits, off, korder, sorter=s)
        _check(bits, off, korder, local=True, sorter=s, perm=perm)
    assert st.passes == H.num_passes(16) + H.segsort_layout(n, len(off) - 1, 16)[3]


@pytest.mark.parametrize("name", sorted(SEGMENTATIONS))
def test_segmentations(name):
    n = (1 << 20) + 13
    off = _offsets(name, n, seed=3)
    rng = np.random.default_rng(4)
    bits = rng.integers(0, 64, n, dtype=np.uint64) * np.uint64(0x0101010101010101)  # heavy ties
    for shape in SHAPES:
        _check(bits, off, 0, flags=shape)
    _check(bits, off, KO.I64 | KO.DESC, local=True)


# ---- 2. radices: sub-digit and digit boundaries of the segment field -----------------------------------------------------
@pytest.mark.parametrize("radix", [8, 11, 13])
@pytest.mark.parametrize("name", ["S255", "S256", "S257", "S65536", "S65537", "len1", "empties"])
def test_radices(radix, name):
    n = 3 * P.PART_TILE + 7 if name != "S65537" else (1 << 18) + 3
    off = _offsets(name, n, seed=radix)
    bits = KO.special_mix(n, seed=radix)
    for shape in SHAPES:
        _check(bits, off, KO.F64, flags=shape, radix=radix)
    _check(bits, off, KO.F64 | KO.DESC, radix=radix, local=True)


# ---- 3. the skip rule: same output with and without NO_SKIP, the expected counts ------------------------------------------
@pytest.mark.parametrize("S", [2, 256, 257, 65536])
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("radix", [8, 16])
def test_no_skip(S, shape, radix):
    n = (1 << 20) + 13
    off = ragged_offsets(np.random.default_rng(S), n, S)
    bits = np.random.default_rng(1).integers(0, 1 << 64, n, dtype=np.uint64) >> np.uint64(8)  # top byte constant
    idxbits, segbits, segw, passes, _ = H.segsort_layout(n, S, radix)
    words = segment_ids(off, n).astype(np.uint64) | (np.arange(n, dtype=np.uint64) << np.uint64(segw))  # retagged keys
    out = []
    for ns in (0, NS):
        flags = shape | ns
        st, _ = _check(bits, off, KO.I64, flags=flags, radix=radix)
        want = (_expected_skips(KO.order_key(bits, KO.I64), flags, radix)
                + _expected_skips(words, flags, radix, passes=range(passes)))
        assert st.passes == H.num_passes(radix) + passes
        assert st.skipped == want, (S, shape, radix, ns, st.skipped, want)
        out.append(st)
    assert out[1].skipped == 0


# ---- 4. special values and structured keys inside ragged segments --------------------------------------------------------
@pytest.mark.parametrize("order", ["f64", "f64_desc"])
def test_special_values(order):
    n = (1 << 20) + 13
    bits = KO.special_mix(n, seed=9)
    for name in ("ragged", "empties", "S257"):
        _check(bits, _offsets(name, n, seed=9), KO.ORDERS[order])


@pytest.mark.parametrize("pattern", P.PATTERNS)
def test_patterns(pattern):
    n = 3 * P.PART_TILE + 7
    bits = np.ascontiguousarray(P.make(pattern, n)["key"])
    _check(bits, _offsets("ragged", n, seed=5), 0)
    _check(bits, _offsets("S256", n, seed=5), KO.I64, flags=TL)


# ---- 5. values: gathered bit for bit, views, aliasing ---------------------------------------------------------------------
@pytest.mark.parametrize("vdtype", [torch.int64, torch.float64])
def test_vals_gathered(vdtype):
    n = (1 << 20) + 13
    off = _offsets("ragged", n, seed=6)
    bits = KO.special_mix(n, seed=6)
    rng = np.random.default_rng(6)
    vals = torch.from_numpy(rng.integers(-(1 << 63), (1 << 63) - 1, n, dtype=np.int64)).cuda().view(vdtype)
    for shape in SHAPES:
        _check(bits, off, KO.F64, flags=shape, vals=vals)
    _check(bits, off, KO.F64, vals=vals, local=True)  # vals win over local_index


def test_views_and_aliasing():
    n = 100003
    off = _offsets("ragged", n, seed=7)
    bits = KO.special_mix(n, seed=7)
    perm = _reference(bits, off, KO.I64)
    kbig = _dev(np.concatenate([np.zeros(1, dtype=np.uint64), bits]), torch.int64)
    vbig = torch.arange(n + 1, device="cuda", dtype=torch.int64) * 3
    obig = torch.from_numpy(np.concatenate([[0], off])).cuda()
    with lsb.DistributedSorter(n, ranks=1, flags=KO.I64) as s:
        k, v, _ = s.sort_segments(kbig[1:], obig[1:], vbig[1:])  # 8-byte aligned views
        assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), 3 * (perm + 1))
        keys = _dev(bits, torch.int64)
        k, v, _ = s.sort_segments(keys, obig[1:], keys_out=keys)  # in place
        assert k.data_ptr() == keys.data_ptr() and np.array_equal(_bits(keys), bits[perm])
        assert np.array_equal(v.cpu().numpy(), perm)
        k, v, _ = s.sort_segments(_dev(bits, torch.int64), obig[1:], vals_out=False)
        assert v is None and np.array_equal(_bits(k), bits[perm])
        k, v, _ = s.sort_segments(_dev(bits, torch.int64), obig[1:], keys_out=False, local_index=True)
        assert k is None and np.array_equal(v.cpu().numpy(), perm - off[segment_ids(off, n)[perm]])


# ---- 6. refusals at the C level ---------------------------------------------------------------------------------------------
def test_c_level_refusals():
    n = 10007
    bits = KO.special_mix(n, seed=12)
    off = _offsets("ragged", n, seed=12)
    keys = _dev(bits, torch.int64)
    out = torch.empty(2 * n, dtype=torch.int64, device="cuda")
    vin = torch.arange(n, device="cuda")
    offs = torch.from_numpy(off).cuda()
    S = len(off) - 1
    with lsb.DistributedSorter(n, ranks=1, flags=KO.I64) as s:
        Lb, ctx = s._L, s._ctx
        p = lambda t: t.data_ptr()  # noqa: E731

        def call(ko, vi, kout, vout, count=n, o=p(offs), nseg=S, flags=0):
            return Lb.lsb_sort_segments_device(ctx, ko, vi, kout, vout, count, o, nseg, flags, None, None)

        sentinel = out.clone()
        assert call(p(keys), None, p(out), None, nseg=0) == ERR_ARG
        assert call(p(keys), None, p(out), None, nseg=-1) == ERR_ARG
        assert call(p(keys), None, p(out), None, flags=2) == ERR_ARG
        assert call(p(keys), None, p(out), None, count=n - 1) == ERR_ARG
        for bad in (off + np.where(np.arange(S + 1) == 0, 1, 0),            # offsets[0] != 0
                    np.where(np.arange(S + 1) == S, n - 1, off),            # offsets[S] != count
                    np.where(np.arange(S + 1) == S // 2, off[S // 2 + 1] + 1, off)):  # decreasing
            bad_t = torch.from_numpy(np.ascontiguousarray(bad, dtype=np.int64)).cuda()
            assert call(p(keys), None, p(out), None, o=p(bad_t)) == ERR_ARG
        assert torch.equal(out, sentinel)  # refused before any key was read or output written
        assert call(p(keys), None, p(out), p(out[n // 2:])) == ERR_ARG    # outputs overlap
        assert call(p(keys), p(vin), p(out), p(vin)) == ERR_ARG           # vals_out overlaps vals_in
        assert call(p(keys), p(vin), p(vin), p(out)) == ERR_ARG           # keys_out overlaps vals_in
        assert call(p(keys), None, p(offs), None) == ERR_ARG              # keys_out overlaps the offsets
        assert call(p(keys), None, p(out), p(offs)) == ERR_ARG            # vals_out overlaps the offsets
        assert call(p(keys), None, None, None) == ERR_ARG                 # no output
        assert call(p(keys), None, p(out), None, nseg=(1 << 48) + 1) == ERR_ARG  # 64 + 14 bits: does not fit
        assert call(None, None, None, None, count=0) == ERR_ARG           # count != here
        st = L.Stats()
        assert Lb.lsb_sort_segments_device(ctx, p(keys), None, p(out), p(out[n:]), n, p(offs), S, 0, None,
                                           ctypes.byref(st)) == 0      # still usable after every refusal
        perm = _reference(bits, off, KO.I64)
        assert np.array_equal(_bits(out[:n]), bits[perm]) and np.array_equal(out[n:].cpu().numpy(), perm)
    with lsb.DistributedSorter(16, ranks=1, radix_bits=13) as s:  # 13 * ceil(53 / 13) = 65 bits of segment id
        k = torch.zeros(16, dtype=torch.uint64, device="cuda")
        o = torch.tensor([0, 16], device="cuda")
        assert s._L.lsb_sort_segments_device(s._ctx, k.data_ptr(), None, k.data_ptr(), None, 16, o.data_ptr(),
                                             (1 << 52) + 1, 0, None, None) == ERR_ARG
    with lsb.DistributedSorter(2 * n, world_size=2, world_rank=0) as s:  # one GPU only, refused before the comm state
        k = torch.zeros(n, dtype=torch.uint64, device="cuda")
        o = torch.tensor([0, n], device="cuda")
        assert s._L.lsb_sort_segments_device(s._ctx, k.data_ptr(), None, k.data_ptr(), None, n, o.data_ptr(), 1, 0,
                                             None, None) == ERR_ARG
        assert "one GPU" in s._L.lsb_last_error(s._ctx).decode()


def test_count_zero_looks_at_no_pointer():
    with lsb.DistributedSorter(0, ranks=1) as s:
        st = L.Stats()
        assert s._L.lsb_sort_segments_device(s._ctx, None, None, None, None, 0, None, 5, 0, None, ctypes.byref(st)) == 0
        assert st.elements == 0 and st.passes == H.num_passes(16) + 1


# ---- 7. ordering against the caller's stream; a reused sorter; one segment == lsb_sort_device -----------------------------
def test_waits_for_the_callers_stream():
    n = (1 << 20) + 7
    bits = KO.special_mix(n, seed=11)
    off = _offsets("ragged", n, seed=11)
    new = _dev(bits, torch.float64)
    keys = torch.zeros(n, dtype=torch.float64, device="cuda")
    offs = torch.zeros(len(off), dtype=torch.int64, device="cuda")
    off_dev = torch.from_numpy(off).cuda()
    side = torch.cuda.Stream()
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64) as s:
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(100_000_000)  # tens of ms on the side stream before the keys and offsets are written
            keys.copy_(new)
            offs.copy_(off_dev)
        k, v, _ = s.sort_segments(keys, offs, stream=side)  # no synchronise in between
    perm = _reference(bits, off, KO.F64)
    assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)


@pytest.mark.parametrize("shape", SHAPES)
def test_reused_sorter_restores_key_order(shape):
    """segment passes sort the segment id as a plain uint64: the context's key order must be back for the next call"""
    n = (1 << 20) + 13
    korder = KO.F64 | KO.DESC
    bits = KO.special_mix(n, seed=13)
    off = _offsets("S257", n, seed=13)
    with lsb.DistributedSorter(n, ranks=1, flags=korder | shape) as s:
        _check(bits, off, korder, sorter=s)
        k, v, _ = s.sort_device(_dev(bits, torch.float64))
        perm = KO.argsort(bits, korder)
        assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)
        _check(bits, off, korder, sorter=s, local=True)
        _check(bits[::-1].copy(), off, korder, sorter=s)


@pytest.mark.parametrize("shape", SHAPES)
def test_one_segment_equals_sort_device(shape):
    n = (1 << 20) + 13
    bits = KO.special_mix(n, seed=14)
    vals = torch.from_numpy(np.random.default_rng(14).standard_normal(n)).cuda()
    with lsb.DistributedSorter(n, ranks=1, flags=KO.F64 | shape) as s:
        for v_in in (None, vals):
            a = s.sort_device(_dev(bits, torch.float64), v_in)
            b = s.sort_segments(_dev(bits, torch.float64), torch.tensor([0, n], device="cuda"), v_in)
            assert torch.equal(a[0].view(torch.int64), b[0].view(torch.int64)) and torch.equal(a[1].view(torch.int64), b[1].view(torch.int64))
            assert a[2].passes == b[2].passes and a[2].skipped == b[2].skipped


# ---- 8. the one-shot forms -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,width", [(1, 100003), (100003, 1), (1024, 1024), (1 << 16, 16), (3, 100003)])
@pytest.mark.parametrize("dtype", [torch.int64, torch.float64])
@pytest.mark.parametrize("descending", [False, True])
def test_rows_equal_torch_sort(rows, width, dtype, descending):
    g = torch.Generator(device="cuda").manual_seed(rows + width)
    if dtype == torch.float64:
        x = torch.randn(rows, width, dtype=dtype, device="cuda", generator=g)
        x[:, ::7] = 0.0
        x[:, 1::11] = -0.0  # -0.0 == +0.0: stable order among zeros
    else:
        x = torch.randint(-50, 50, (rows, width), dtype=dtype, device="cuda", generator=g)  # many ties
    k, i = lsb.sort_segments(x, descending=descending)
    tk, ti = torch.sort(x, dim=-1, stable=True, descending=descending)
    assert k.shape == x.shape and i.shape == x.shape and i.dtype == torch.int64
    assert torch.equal(k.view(torch.int64), tk.view(torch.int64)) and torch.equal(i, ti)
    vals = torch.randn(rows, width, dtype=torch.float64, device="cuda", generator=g)
    k, v = lsb.sort_segments(x, vals=vals, descending=descending)
    assert torch.equal(v.view(torch.int64), vals.gather(1, ti).view(torch.int64))


def test_oneshot_ragged_uint64():
    n = (1 << 20) + 13
    bits = np.random.default_rng(15).integers(0, 1 << 64, n, dtype=np.uint64)
    off = _offsets("empties", n, seed=15)
    k, v = lsb.sort_segments(_dev(bits, torch.uint64), torch.from_numpy(off).cuda())
    perm = _reference(bits, off, 0)
    assert k.dtype == torch.uint64 and np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), perm)
    vals = torch.from_numpy(np.arange(n, dtype=np.int64) * 7).cuda()
    k, v = lsb.sort_segments(_dev(bits, torch.uint64), torch.from_numpy(off).cuda(), vals=vals, descending=True)
    perm = _reference(bits, off, KO.DESC)
    assert np.array_equal(_bits(k), bits[perm]) and np.array_equal(v.cpu().numpy(), 7 * perm)
